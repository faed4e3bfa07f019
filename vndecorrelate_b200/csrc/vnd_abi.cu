// extern "C" surface of libvnd_b200.so (see include/vnd_b200.h): argument checking, the device
// entry points, and the host-buffer entry points with their context (device arena, streams,
// pinned staging).

#include <cuda.h>  // CUcontext / CUresult types only: cuCtxGetCurrent is fetched through cudaGetDriverEntryPoint
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

#include "vnd_batch.cuh"
#include "vnd_common.cuh"

namespace vnd {

// ---- launchers implemented in the kernel translation units ----------------------------------
int sparse_fir_launch(const vnd_signal* x, const vnd_signal* y, const vnd_tap_program* taps, int max_prog_words, cudaStream_t st);
int vn_stereo_launch(const vnd_signal* x, void* out, int out_dtype, long long o_st, long long o_sc, const vnd_tap_program* taps,
                     int prog_words, const vnd_epilogue* ep, const float* gains, int delay, int delay_ch, cudaStream_t st);
int seq_sumsq_launch(const vnd_signal* a, const vnd_signal* b, void* sums, cudaStream_t st);
int colsumsq_launch(const vnd_signal* a, const vnd_signal* b, void* sums, void* leaf, size_t leaf_bytes, cudaStream_t st);
size_t colsumsq_workspace_bytes(long long frames);
int rms_gain_launch(const void* sums, void* gains, int channels, long long frames, int dtype, cudaStream_t st);
int place_launch(const float* y, long long y_st, long long y_sc, long long frames, int channels, const vnd_signal* out,
                 const float* gains, int delay, int delay_ch, cudaStream_t st);
int scale_launch(float* y, long long y_st, long long y_sc, long long frames, int channels, const float* gains, cudaStream_t st);
int haas_launch(const vnd_signal* x, const vnd_signal* out, int delay, int delay_ch, int mode_ms, int mono, int use_width,
                double width, cudaStream_t st);
int stereo_op_launch(const vnd_signal* a, const vnd_signal* dry, int op, double width, const void* gains, cudaStream_t st);
int transpose_launch(const float* src, float* dst, long long rows, long long cols, cudaStream_t st);
int transpose_launch_ld(const float* src, float* dst, long long rows, long long cols, long long ld_src, long long ld_dst, cudaStream_t st);
int objective_workspace_bytes(long long frames, int n_clips, int n_cand, size_t* bytes);
int vn_objective_launch(const float* clips, long long frames, int n_clips, long long clip_stride, long long chan_stride,
                        const vnd_tap_program* cand, double* partials, void* workspace, size_t workspace_bytes, cudaStream_t st);
int haas_objective_launch(const void* clips, int clip_dtype, long long frames, int n_clips, long long clip_stride, long long chan_stride,
                          const int* delays, int n_cand, double* partials, cudaStream_t st);
int objective_runs_workspace_bytes(const long long* offs, const int* run_clip, const int* run_count, int n_runs, size_t* bytes);
int vn_objective_runs_launch(const float* x, long long chan_stride, const long long* offs, const int* run_clip, const int* run_cand,
                             const int* run_count, const int* run_out, int n_runs, const vnd_tap_program* cand, double* partials,
                             void* workspace, size_t workspace_bytes, cudaStream_t st);
int haas_objective_pairs_launch(const float* x, long long chan_stride, const long long* offs, const int* pair_clip, const int* pair_delay,
                                int n_pairs, double* partials, cudaStream_t st);
int haas_effect_objective_launch(const float* x, long long frames, long long chan_stride, const vnd_haas_clip* cands, int n_cand, double* partials,
                                 cudaStream_t st);
int vn_stereo_objective_workspace_bytes(long long frames, int n_cand, size_t* bytes);
int vn_stereo_objective_launch(const float* x, long long frames, long long chan_stride, const vnd_tap_program* taps, const vnd_vn_stereo_cand* cands,
                               int n_cand, double* partials, void* workspace, size_t workspace_bytes, cudaStream_t st);
int vn_stereo_rms_objective_launch(const float* x, long long frames, long long chan_stride, const vnd_tap_program* taps,
                                   const vnd_vn_stereo_cand* cands, int n_cand, float* gains, double* partials, void* workspace,
                                   size_t workspace_bytes, cudaStream_t st);
size_t dsp_workspace_bytes(long long elems);
int rms_normalize_launch(const vnd_signal* x, const vnd_signal* y, int x_ndim, int y_ndim, int stereo_mode, double eps, void* ws, cudaStream_t st);
int peak_normalize_launch(const vnd_signal* y, int ndim, int stereo_mode, double eps, void* ws, cudaStream_t st);
int polar_launch(const void* l, const void* r, long long n, int dtype, int mode_ms, int semicircular, int normalize, void* radii, void* thetas,
                 void* weights, void* ws, cudaStream_t st);

// ---- error state ----------------------------------------------------------------------------
static thread_local char t_error[512] = "";
std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(t_error, sizeof(t_error), fmt, ap);
  va_end(ap);
}

int device_info(DeviceInfo* out) {
  static std::mutex mu;
  static DeviceInfo cache[64];
  static bool have[64] = {false};
  int dev = 0;
  VND_CUDA_OK(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  if (dev < 0 || dev >= 64) dev = 0;
  if (!have[dev]) {
    VND_CUDA_OK(cudaDeviceGetAttribute(&cache[dev].sm_count, cudaDevAttrMultiProcessorCount, dev));
    VND_CUDA_OK(cudaDeviceGetAttribute(&cache[dev].max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    have[dev] = true;
  }
  *out = cache[dev];
  return VND_OK;
}

static int check_signal(const vnd_signal* s, const char* name, bool need_data = true) {
  VND_REQUIRE(s != nullptr, VND_EINVAL, "%s is null", name);
  VND_REQUIRE(s->frames >= 0 && s->channels >= 0, VND_EINVAL, "%s has a negative extent", name);
  VND_REQUIRE(s->dtype == VND_F32 || s->dtype == VND_F64, VND_EINVAL, "%s has an unknown dtype %d", name, s->dtype);
  VND_REQUIRE(!need_data || s->data != nullptr || s->frames * (long long)s->channels == 0, VND_EINVAL, "%s has no data pointer", name);
  return VND_OK;
}

static int check_taps(const vnd_tap_program* t) {
  VND_REQUIRE(t != nullptr, VND_EINVAL, "tap program is null");
  VND_REQUIRE(t->channels >= 0 && t->n_words >= 0, VND_EINVAL, "tap program has a negative extent");
  VND_REQUIRE(t->channels == 0 || t->offsets != nullptr, VND_EPROGRAM, "tap program has no offsets");
  VND_REQUIRE(t->n_words == 0 || t->words != nullptr, VND_EPROGRAM, "tap program has no words");
  VND_REQUIRE(t->order >= VND_ORDER_SEGMENTED && t->order <= VND_ORDER_ASCENDING_F64, VND_EINVAL, "unknown tap order %d", t->order);
  VND_REQUIRE(t->halo >= 0 && t->max_channel_words >= 0, VND_EPROGRAM, "tap program has a negative halo or block size");
  return VND_OK;
}

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace vnd

using namespace vnd;

// ================================================================================================
// housekeeping
// ================================================================================================
extern "C" int vnd_abi_version(void) { return VND_ABI_VERSION; }
extern "C" const char* vnd_version(void) { return "vnd_b200 0.1.0 (sm_100a)"; }
extern "C" const char* vnd_last_error(void) { return t_error; }
extern "C" int64_t vnd_launch_count(void) { return (int64_t)g_launches.load(); }

extern "C" const char* vnd_status_string(int status) {
  switch (status) {
    case VND_OK: return "ok";
    case VND_EINVAL: return "invalid argument";
    case VND_ECUDA: return "CUDA runtime error";
    case VND_EUNSUPPORTED: return "unsupported request";
    case VND_ENOMEM: return "workspace or memory too small";
    case VND_EPROGRAM: return "malformed tap program";
    default: return "unknown status";
  }
}

extern "C" int vnd_device_count(int* count) {
  VND_REQUIRE(count != nullptr, VND_EINVAL, "count is null");
  *count = 0;
  VND_CUDA_OK(cudaGetDeviceCount(count));
  return VND_OK;
}

// ================================================================================================
// device entry points
// ================================================================================================
static int check_sparse_fir(const vnd_signal* x, const vnd_signal* y, const vnd_tap_program* taps) {
  int rc;
  if ((rc = check_signal(x, "x")) || (rc = check_signal(y, "y")) || (rc = check_taps(taps))) return rc;
  VND_REQUIRE(y->dtype == VND_F32, VND_EINVAL, "y must be float32 (the reference's output buffers are float32)");
  VND_REQUIRE(y->frames == x->frames, VND_EINVAL, "x has %lld frames but y has %lld", (long long)x->frames, (long long)y->frames);
  VND_REQUIRE(y->channels == taps->channels, VND_EINVAL, "y has %d channels but the tap program has %d", y->channels, taps->channels);
  VND_REQUIRE(x->channels >= taps->channels || x->stride_c == 0, VND_EINVAL, "x has %d channels, fewer than the %d outputs",
              x->channels, taps->channels);
  return VND_OK;
}

extern "C" int vnd_sparse_fir_dev(const vnd_signal* x, const vnd_signal* y, const vnd_tap_program* taps, void* stream) {
  int rc;
  if ((rc = check_sparse_fir(x, y, taps))) return rc;
  return sparse_fir_launch(x, y, taps, taps->max_channel_words, (cudaStream_t)stream);
}

extern "C" int vnd_vn_decorrelate_workspace(int64_t frames, int32_t channels, const vnd_epilogue* ep, size_t* bytes) {
  VND_REQUIRE(bytes != nullptr && ep != nullptr, VND_EINVAL, "null argument");
  VND_REQUIRE(frames >= 0 && channels >= 0, VND_EINVAL, "negative extent");
  // status words | sums and gains | leaf sums of the pairwise order (planar inputs) | float32 scratch of the result
  *bytes = 256 + align_up((size_t)channels * 3 * sizeof(float), 256) + align_up(colsumsq_workspace_bytes(frames), 256) +
           (size_t)frames * channels * sizeof(float);
  return VND_OK;
}

static int check_vn_decorrelate(const vnd_signal* x, const vnd_signal* out, const vnd_tap_program* taps, const vnd_epilogue* ep) {
  int rc;
  if ((rc = check_signal(x, "x")) || (rc = check_signal(out, "out")) || (rc = check_taps(taps))) return rc;
  VND_REQUIRE(ep != nullptr, VND_EINVAL, "epilogue is null");
  VND_REQUIRE(x->dtype == VND_F32, VND_EINVAL, "x must be float32 (decorrelate casts first, decorrelation.py:426)");
  VND_REQUIRE(taps->order == VND_ORDER_SEGMENTED, VND_EINVAL, "decorrelate needs a SEGMENTED tap program");
  const int C = taps->channels;
  VND_REQUIRE(ep->haas_delay >= 0, VND_EINVAL, "negative Haas delay");
  VND_REQUIRE(out->channels == C, VND_EINVAL, "out has %d channels but the tap program has %d", out->channels, C);
  VND_REQUIRE(out->frames == x->frames + ep->haas_delay, VND_EINVAL, "out must have frames + haas_delay = %lld frames, has %lld",
              (long long)x->frames + ep->haas_delay, (long long)out->frames);
  VND_REQUIRE(x->channels >= C || x->stride_c == 0, VND_EINVAL, "x has fewer channels than the program");
  if (ep->ms_encode || ep->use_width || ep->haas_delay > 0)
    VND_REQUIRE(C == 2, VND_EINVAL, "M/S encode, width and the Haas delay need exactly 2 channels (utils/dsp.py:297-302)");
  if (ep->haas_delay > 0) VND_REQUIRE(ep->haas_channel == 0 || ep->haas_channel == 1, VND_EINVAL, "haas_channel must be 0 or 1");
  return VND_OK;
}

extern "C" int vnd_vn_decorrelate_dev(const vnd_signal* x, const vnd_signal* out, const vnd_tap_program* taps,
                                      const vnd_epilogue* ep, void* workspace, size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_vn_decorrelate(x, out, taps, ep))) return rc;
  const int C = taps->channels;
  const long long L = x->frames;
  cudaStream_t st = (cudaStream_t)stream;
  const int delay = ep->haas_delay, dch = ep->haas_channel;

  size_t need = 0;
  vnd_vn_decorrelate_workspace(L, C, ep, &need);
  char* ws = reinterpret_cast<char*>(workspace);
  float* sums = reinterpret_cast<float*>(ws);
  float* gains = sums + 2 * (size_t)C;
  char* leaf = ws + align_up((size_t)C * 3 * sizeof(float), 256);
  const size_t leaf_bytes = align_up(colsumsq_workspace_bytes(L), 256);
  float* scratch = reinterpret_cast<float*>(leaf + leaf_bytes);

  if (L == 0 || C == 0) return place_launch(nullptr, 0, 0, 0, C, out, nullptr, delay, dch, st);

  // one kernel, one read and one write per sample
  if (!ep->rms_normalize && C == 2) {
    rc = vn_stereo_launch(x, out->data, out->dtype, out->stride_t, out->stride_c, taps, taps->max_channel_words * 2, ep, nullptr,
                          delay, dch, st);
    if (rc != VND_EUNSUPPORTED) return rc;
  }
  VND_REQUIRE(workspace != nullptr && workspace_bytes >= need, VND_ENOMEM, "workspace too small: need %zu bytes, have %zu", need,
              workspace_bytes);
  vnd_signal y{scratch, L, C, VND_F32, C, 1};
  rc = VND_EUNSUPPORTED;
  if (C == 2) rc = vn_stereo_launch(x, scratch, VND_F32, 2, 1, taps, taps->max_channel_words * 2, ep, nullptr, 0, 0, st);
  if (rc == VND_EUNSUPPORTED) {  // unfused composition (halo too long for the stereo kernel, or C != 2)
    if ((rc = sparse_fir_launch(x, &y, taps, taps->max_channel_words, st))) return rc;
    if (ep->ms_encode && (rc = stereo_op_launch(&y, x, 3, 0.0, nullptr, st))) return rc;
    if (ep->use_width && (rc = stereo_op_launch(&y, nullptr, 2, ep->width, nullptr, st))) return rc;
  } else if (rc) {
    return rc;
  }
  const float* g = nullptr;
  if (ep->rms_normalize) {
    vnd_signal xa = *x;
    xa.channels = C;
    if ((rc = colsumsq_launch(&xa, &y, sums, leaf, leaf_bytes, st))) return rc;  // x in the order its layout gives it in numpy
    if ((rc = rms_gain_launch(sums, gains, C, L, VND_F32, st))) return rc;
    g = gains;
  }
  return place_launch(scratch, C, 1, L, C, out, g, delay, dch, st);
}

// Arguments of the batched decorrelate that can be checked without reading device memory.
static int check_batch(const void* x, int32_t x_dtype, int64_t rows, const void* offsets, int32_t n_clips, const void* program_of_clip,
                       const vnd_tap_program* taps, const vnd_epilogue* ep, const void* out, int32_t out_dtype) {
  int rc;
  VND_REQUIRE(rows >= 0 && n_clips >= 0, VND_EINVAL, "negative extent (rows %lld, n_clips %d)", (long long)rows, n_clips);
  VND_REQUIRE(n_clips > 0 || rows == 0, VND_EINVAL, "%lld rows but no clips", (long long)rows);
  VND_REQUIRE(x_dtype == VND_F32, VND_EINVAL, "the packed input must be float32 (decorrelate casts first, decorrelation.py:426)");
  VND_REQUIRE(out_dtype == VND_F32 || out_dtype == VND_F64, VND_EINVAL, "unknown output dtype %d", out_dtype);
  VND_REQUIRE(ep != nullptr, VND_EINVAL, "epilogue is null");
  VND_REQUIRE(ep->haas_delay >= 0, VND_EINVAL, "negative Haas delay");
  if (ep->haas_delay > 0) VND_REQUIRE(ep->haas_channel == 0 || ep->haas_channel == 1, VND_EINVAL, "haas_channel must be 0 or 1");
  if ((rc = check_taps(taps))) return rc;
  VND_REQUIRE(taps->order == VND_ORDER_SEGMENTED, VND_EINVAL, "decorrelate needs a SEGMENTED tap program");
  VND_REQUIRE(taps->channels % 2 == 0, VND_EINVAL, "the tap program has %d channels: it must hold two per filter", taps->channels);
  VND_REQUIRE(n_clips == 0 || taps->channels >= 2, VND_EINVAL, "the tap program holds no filter");
  VND_REQUIRE(x != nullptr || rows == 0, VND_EINVAL, "x is null");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(x) % 8 == 0, VND_EINVAL, "x must be 8-byte aligned (one float32 pair per row)");
  VND_REQUIRE((offsets != nullptr && program_of_clip != nullptr) || n_clips == 0, VND_EINVAL, "frame_offsets or program_of_clip is null");
  VND_REQUIRE(out != nullptr || rows + (long long)n_clips * ep->haas_delay == 0, VND_EINVAL, "out is null");
  return VND_OK;
}

// Does the batched stereo kernel hold tile + halo of this program?
static bool batch_fits(const vnd_tap_program* taps, int64_t rows) {
  long long halo = taps->halo > 0 ? taps->halo : 0;
  if (halo > rows) halo = rows;
  size_t smem = 0;
  return vn_batch_smem((int)halo, 2 * taps->max_channel_words, &smem);
}

extern "C" int vnd_vn_decorrelate_batch_workspace(int64_t rows, int32_t n_clips, const vnd_epilogue* ep, size_t* bytes) {
  VND_REQUIRE(bytes != nullptr && ep != nullptr, VND_EINVAL, "null argument");
  VND_REQUIRE(rows >= 0 && n_clips >= 0, VND_EINVAL, "negative extent");
  *bytes = vn_batch_workspace_bytes(rows, n_clips, ep->rms_normalize);
  return VND_OK;
}

extern "C" int vnd_vn_decorrelate_batch_dev(const void* x, int32_t x_dtype, int64_t rows, const int64_t* frame_offsets, int32_t n_clips,
                                            const int32_t* program_of_clip, const vnd_tap_program* taps, const vnd_epilogue* ep, void* out,
                                            int32_t out_dtype, void* workspace, size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_batch(x, x_dtype, rows, frame_offsets, n_clips, program_of_clip, taps, ep, out, out_dtype))) return rc;
  if (n_clips == 0) return VND_OK;
  VND_REQUIRE(batch_fits(taps, rows), VND_EUNSUPPORTED,
              "a halo of %d frames does not fit the batched kernel; run these clips through vnd_vn_decorrelate_dev", taps->halo);
  const size_t need = vn_batch_workspace_bytes(rows, n_clips, ep->rms_normalize);
  VND_REQUIRE(need == 0 || (workspace != nullptr && workspace_bytes >= need), VND_ENOMEM, "workspace too small: need %zu bytes, have %zu",
              need, workspace_bytes);
  VND_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 16 == 0, VND_EINVAL, "workspace must be 16-byte aligned");
  return vn_batch_launch(reinterpret_cast<const float*>(x), rows, reinterpret_cast<const long long*>(frame_offsets), n_clips,
                         program_of_clip, taps, ep, out, out_dtype, workspace, (cudaStream_t)stream);
}

extern "C" int vnd_colsumsq_seq_f32_dev(const vnd_signal* a, float* sums, void* stream) {
  int rc;
  if ((rc = check_signal(a, "a"))) return rc;
  VND_REQUIRE(a->dtype == VND_F32, VND_EINVAL, "a must be float32");
  VND_REQUIRE(sums != nullptr || a->channels == 0, VND_EINVAL, "sums is null");
  return seq_sumsq_launch(a, nullptr, sums, (cudaStream_t)stream);
}

static int check_haas(const vnd_signal* x, const vnd_signal* out, int32_t delay, int32_t delayed_channel) {
  int rc;
  if ((rc = check_signal(x, "x")) || (rc = check_signal(out, "out"))) return rc;
  VND_REQUIRE(x->dtype == VND_F32 && out->dtype == VND_F64, VND_EINVAL, "Haas takes float32 in and float64 out (decorrelation.py:194,206)");
  VND_REQUIRE(delay >= 0, VND_EINVAL, "negative delay");
  VND_REQUIRE(delayed_channel == 0 || delayed_channel == 1, VND_EINVAL, "delayed_channel must be 0 or 1");
  VND_REQUIRE(out->channels == 2 && out->frames == x->frames + delay, VND_EINVAL, "out must be (frames + delay, 2)");
  return VND_OK;
}

extern "C" int vnd_haas_dev(const vnd_signal* x, const vnd_signal* out, int32_t delay, int32_t delayed_channel, int32_t mode_ms,
                            int32_t mono, int32_t use_width, double width, void* stream) {
  int rc;
  if ((rc = check_haas(x, out, delay, delayed_channel))) return rc;
  return haas_launch(x, out, delay, delayed_channel, mode_ms, mono, use_width, width, (cudaStream_t)stream);
}

// Arguments of the batched Haas effect that can be checked without reading the tables.
static int check_haas_batch(const float* x, int64_t rows, const void* frame_offsets, int32_t n_clips, const vnd_haas_clip* clips) {
  VND_REQUIRE(rows >= 0 && n_clips >= 0, VND_EINVAL, "negative extent (rows %lld, n_clips %d)", (long long)rows, n_clips);
  VND_REQUIRE(n_clips > 0 || rows == 0, VND_EINVAL, "%lld rows but no clips", (long long)rows);
  VND_REQUIRE(x != nullptr || rows == 0, VND_EINVAL, "x is null");
  VND_REQUIRE((frame_offsets != nullptr && clips != nullptr) || n_clips == 0, VND_EINVAL, "frame_offsets or clips is null");
  return VND_OK;
}

extern "C" int vnd_haas_batch_dev(const float* x, int64_t rows, const int64_t* frame_offsets, int32_t n_clips, const vnd_haas_clip* clips,
                                  const int64_t* out_offsets, int64_t out_rows, double* out, void* stream) {
  int rc;
  if ((rc = check_haas_batch(x, rows, frame_offsets, n_clips, clips))) return rc;
  VND_REQUIRE(out_rows >= rows, VND_EINVAL, "out_rows = %lld is less than rows = %lld", (long long)out_rows, (long long)rows);
  VND_REQUIRE(out_offsets != nullptr || n_clips == 0, VND_EINVAL, "out_offsets is null");
  VND_REQUIRE(out != nullptr || out_rows == 0, VND_EINVAL, "out is null");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(x) % 8 == 0, VND_EINVAL, "x must be 8-byte aligned (one float32 pair per row)");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(clips) % 16 == 0, VND_EINVAL, "clips must be 16-byte aligned");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(out) % 16 == 0, VND_EINVAL, "out must be 16-byte aligned (one float64 pair per row)");
  return haas_batch_launch(x, reinterpret_cast<const long long*>(frame_offsets), n_clips, clips, reinterpret_cast<const long long*>(out_offsets),
                           out_rows, out, (cudaStream_t)stream);
}

// Arguments of a block step that can be checked without reading device memory; fills the step's tables.  x and the
// history buffers hold `align`-byte values (a float32 pair per row for the stereo steps).
static int check_block_step(const void* x, int64_t rows, const int64_t* frame_offsets, int32_t n_signals, const int64_t* received,
                            const void* history_in, void* history_out, int32_t history_frames, const int64_t* out_offsets,
                            int64_t out_rows, const void* out, int align, BlockStepParams* b) {
  VND_REQUIRE(rows >= 0 && n_signals >= 0 && out_rows >= 0 && history_frames >= 0, VND_EINVAL,
              "negative extent (rows %lld, n_signals %d, out_rows %lld, history_frames %d)", (long long)rows, n_signals, (long long)out_rows,
              history_frames);
  VND_REQUIRE(n_signals > 0 || rows + out_rows == 0, VND_EINVAL, "%lld rows and %lld out rows but no signals", (long long)rows,
              (long long)out_rows);
  VND_REQUIRE(x != nullptr || rows == 0, VND_EINVAL, "x is null");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(x) % align == 0, VND_EINVAL, "x must be %d-byte aligned", align);
  VND_REQUIRE((frame_offsets != nullptr && received != nullptr && out_offsets != nullptr) || n_signals == 0, VND_EINVAL,
              "frame_offsets, received or out_offsets is null");
  VND_REQUIRE(out != nullptr || out_rows == 0, VND_EINVAL, "out is null");
  const bool hist = history_frames > 0 && n_signals > 0;
  VND_REQUIRE(!hist || (history_in != nullptr && history_out != nullptr), VND_EINVAL, "a history buffer is null");
  VND_REQUIRE(!hist || history_in != history_out, VND_EINVAL, "history_in and history_out must be two buffers");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(history_in) % align == 0 && reinterpret_cast<uintptr_t>(history_out) % align == 0, VND_EINVAL,
              "the history buffers must be %d-byte aligned", align);
  *b = BlockStepParams{};
  b->x = x;
  b->offs = reinterpret_cast<const long long*>(frame_offsets);
  b->received = reinterpret_cast<const long long*>(received);
  b->out_offs = reinterpret_cast<const long long*>(out_offsets);
  b->hist_in = history_in;
  b->hist_out = history_out;
  b->n = n_signals;
  b->H = history_frames;
  b->C = 2;
  return VND_OK;
}

extern "C" int vnd_vn_block_step_dev(const float* x, int64_t rows, const int64_t* frame_offsets, int32_t n_signals, const int64_t* received,
                                     const int64_t* emitted, const int32_t* program_of_signal, const vnd_tap_program* taps,
                                     const vnd_epilogue* ep, const float* history_in, float* history_out, int32_t history_frames,
                                     const int64_t* out_offsets, int64_t out_rows, float* out, void* stream) {
  int rc;
  if ((rc = check_taps(taps))) return rc;
  VND_REQUIRE(taps->order == VND_ORDER_SEGMENTED, VND_EINVAL, "decorrelate needs a SEGMENTED tap program");
  VND_REQUIRE(taps->channels % 2 == 0, VND_EINVAL, "the tap program has %d channels: it must hold two per filter", taps->channels);
  VND_REQUIRE(ep != nullptr, VND_EINVAL, "epilogue is null");
  VND_REQUIRE(!ep->rms_normalize, VND_EINVAL, "rms_normalize depends on the whole signal and cannot run block by block");
  VND_REQUIRE(ep->haas_delay == 0, VND_EINVAL, "the Haas stage of a block step is vnd_haas_block_step_dev");
  size_t smem = 0;
  VND_REQUIRE(vn_batch_smem(((taps->halo > 0 ? taps->halo : 0) + 3) & ~3, 2 * taps->max_channel_words, &smem), VND_EUNSUPPORTED,
              "a halo of %d frames does not fit the block-step kernel's shared memory", taps->halo);
  VND_REQUIRE(history_frames >= taps->halo - 1, VND_EINVAL, "%d history frames cannot hold the %d frames the filter reads ahead",
              history_frames, taps->halo - 1);
  BlockStepParams b;
  if ((rc = check_block_step(x, rows, frame_offsets, n_signals, received, history_in, history_out, history_frames, out_offsets, out_rows, out,
                             8, &b)))
    return rc;
  VND_REQUIRE(n_signals == 0 || taps->channels >= 2, VND_EINVAL, "the tap program holds no filter");
  VND_REQUIRE((emitted != nullptr && program_of_signal != nullptr) || n_signals == 0, VND_EINVAL, "emitted or program_of_signal is null");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(out) % 8 == 0, VND_EINVAL, "out must be 8-byte aligned (one float32 pair per row)");
  if (n_signals == 0 || rows + out_rows == 0) return VND_OK;
  b.emitted = reinterpret_cast<const long long*>(emitted);
  return vn_block_step_launch(b, out_rows, program_of_signal, taps, ep, out, (cudaStream_t)stream);
}

extern "C" int vnd_haas_block_step_dev(const float* x, int64_t rows, const int64_t* frame_offsets, int32_t n_signals, const int64_t* received,
                                       const vnd_haas_clip* signals, const float* history_in, float* history_out, int32_t history_frames,
                                       const int64_t* out_offsets, int64_t out_rows, double* out, void* stream) {
  int rc;
  BlockStepParams b;
  if ((rc = check_block_step(x, rows, frame_offsets, n_signals, received, history_in, history_out, history_frames, out_offsets, out_rows, out,
                             8, &b)))
    return rc;
  VND_REQUIRE(signals != nullptr || n_signals == 0, VND_EINVAL, "signals is null");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(signals) % 16 == 0, VND_EINVAL, "signals must be 16-byte aligned");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(out) % 16 == 0, VND_EINVAL, "out must be 16-byte aligned (one float64 pair per row)");
  if (n_signals == 0 || rows + out_rows == 0) return VND_OK;
  return haas_block_step_launch(b, out_rows, signals, out, (cudaStream_t)stream);
}

extern "C" int vnd_fir_block_step_dev(const void* x, int32_t dtype, int64_t rows, int32_t channels, const int64_t* frame_offsets,
                                      int32_t n_signals, const int64_t* received, const int64_t* emitted, const int32_t* program_of_signal,
                                      const vnd_tap_program* taps, const void* history_in, void* history_out, int32_t history_frames,
                                      const int64_t* out_offsets, int64_t out_rows, float* out, void* stream) {
  int rc;
  if ((rc = check_taps(taps))) return rc;
  VND_REQUIRE(taps->order == VND_ORDER_SEGMENTED, VND_EINVAL, "convolve needs a SEGMENTED tap program");
  VND_REQUIRE(dtype == VND_F32 || dtype == VND_F64, VND_EINVAL, "unknown dtype %d", dtype);
  VND_REQUIRE(channels > 0, VND_EINVAL, "channels must be positive, got %d", channels);
  VND_REQUIRE(taps->channels % channels == 0, VND_EINVAL, "the tap program has %d channels: it must hold %d per filter", taps->channels,
              channels);
  VND_REQUIRE(history_frames >= taps->halo - 1, VND_EINVAL, "%d history frames cannot hold the %d frames the filter reads ahead",
              history_frames, taps->halo - 1);
  BlockStepParams b;
  const int elem = dtype == VND_F64 ? 8 : 4;
  if ((rc = check_block_step(x, rows, frame_offsets, n_signals, received, history_in, history_out, history_frames, out_offsets, out_rows, out,
                             elem, &b)))
    return rc;
  VND_REQUIRE(n_signals == 0 || taps->channels >= channels, VND_EINVAL, "the tap program holds no filter");
  VND_REQUIRE((emitted != nullptr && program_of_signal != nullptr) || n_signals == 0, VND_EINVAL, "emitted or program_of_signal is null");
  VND_REQUIRE(reinterpret_cast<uintptr_t>(out) % 4 == 0, VND_EINVAL, "out must be 4-byte aligned");
  if (n_signals == 0 || rows + out_rows == 0) return VND_OK;
  b.emitted = reinterpret_cast<const long long*>(emitted);
  b.C = channels;
  return fir_block_step_launch(b, out_rows, dtype, program_of_signal, taps, out, (cudaStream_t)stream);
}

static int check_stereo_op(const vnd_signal* a, const vnd_signal* dry, int32_t op) {
  int rc;
  if ((rc = check_signal(a, "a"))) return rc;
  VND_REQUIRE(op >= 0 && op <= 4, VND_EINVAL, "unknown stereo op %d", op);
  VND_REQUIRE(a->channels == 2, VND_EINVAL, "stereo helpers need a (frames, 2) signal (utils/dsp.py:297-302)");
  if (op == 3 || op == 4) {
    if ((rc = check_signal(dry, "dry"))) return rc;
    VND_REQUIRE(dry->channels == 2 && dry->frames == a->frames && dry->dtype == a->dtype, VND_EINVAL,
                "dry must match a in shape and dtype");
  }
  return VND_OK;
}

extern "C" int vnd_stereo_op_dev(const vnd_signal* a, const vnd_signal* dry, int32_t op, double width, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_stereo_op(a, dry, op))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (op == 4) {
    const size_t esz = a->dtype == VND_F64 ? 8 : 4;
    VND_REQUIRE(workspace != nullptr && workspace_bytes >= 64, VND_ENOMEM, "rms workspace needs at least 64 bytes");
    char* sums = reinterpret_cast<char*>(workspace);
    char* gains = sums + 4 * esz;
    // planar (Fortran-ordered) signals are summed in numpy's pairwise order and need 64 + 8 (frames / 64 + 8) bytes
    if ((rc = colsumsq_launch(dry, a, sums, sums + 64, workspace_bytes - 64, st))) return rc;
    if ((rc = rms_gain_launch(sums, gains, 2, a->frames, a->dtype, st))) return rc;
    return stereo_op_launch(a, nullptr, 4, 0.0, gains, st);
  }
  return stereo_op_launch(a, op == 3 ? dry : nullptr, op, width, nullptr, st);
}

extern "C" int vnd_objective_workspace(int64_t frames, int32_t n_clips, int32_t n_cand, size_t* bytes) {
  VND_REQUIRE(bytes != nullptr, VND_EINVAL, "bytes is null");
  VND_REQUIRE(frames >= 0 && n_clips >= 0 && n_cand >= 0, VND_EINVAL, "negative extent");
  return objective_workspace_bytes(frames, n_clips, n_cand, bytes);
}

static int check_vn_objective_batch(const float* clips, int64_t frames, int32_t n_clips, const vnd_tap_program* cand, const double* partials) {
  int rc;
  if ((rc = check_taps(cand))) return rc;
  VND_REQUIRE(cand->order == VND_ORDER_SEGMENTED, VND_EINVAL, "objective candidates need SEGMENTED tap programs");
  VND_REQUIRE(frames >= 0 && n_clips >= 0, VND_EINVAL, "negative extent");
  if (n_clips == 0 || cand->channels == 0) return VND_OK;
  VND_REQUIRE(clips != nullptr && partials != nullptr, VND_EINVAL, "null buffer");
  // the reference takes max(|theta|) of the frames: an empty signal is a ValueError there (optimization.py:41-43)
  VND_REQUIRE(frames > 0, VND_EINVAL, "objective of an empty signal (zero-size array to reduction operation maximum which has no identity)");
  return VND_OK;
}

extern "C" int vnd_vn_objective_batch_dev(const float* clips, int64_t frames, int32_t n_clips, int64_t clip_stride, int64_t chan_stride,
                                          const vnd_tap_program* cand, double* partials, void* workspace, size_t workspace_bytes,
                                          void* stream) {
  int rc;
  if ((rc = check_vn_objective_batch(clips, frames, n_clips, cand, partials))) return rc;
  return vn_objective_launch(clips, frames, n_clips, clip_stride, chan_stride, cand, partials, workspace, workspace_bytes,
                             (cudaStream_t)stream);
}

static int check_haas_objective_batch(const void* clips, int32_t clip_dtype, int64_t frames, int32_t n_clips, const int32_t* delays,
                                      int32_t n_cand, const double* partials) {
  VND_REQUIRE(frames >= 0 && n_clips >= 0 && n_cand >= 0, VND_EINVAL, "negative extent");
  VND_REQUIRE((clips != nullptr && partials != nullptr && delays != nullptr) || n_clips == 0 || n_cand == 0, VND_EINVAL, "null buffer");
  VND_REQUIRE(clip_dtype == VND_F32 || clip_dtype == VND_F64, VND_EINVAL, "unknown clip dtype %d", clip_dtype);
  return VND_OK;
}

extern "C" int vnd_haas_objective_batch_dev(const void* clips, int32_t clip_dtype, int64_t frames, int32_t n_clips, int64_t clip_stride,
                                            int64_t chan_stride, const int32_t* delays, int32_t n_cand, double* partials, void* workspace,
                                            size_t workspace_bytes, void* stream) {
  (void)workspace;
  (void)workspace_bytes;
  int rc;
  if ((rc = check_haas_objective_batch(clips, clip_dtype, frames, n_clips, delays, n_cand, partials))) return rc;
  return haas_objective_launch(clips, clip_dtype, frames, n_clips, clip_stride, chan_stride, delays, n_cand, partials, (cudaStream_t)stream);
}

// Arguments of the pair-list Haas objective that can be checked without reading device memory.
static int check_haas_pairs(const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets, int32_t n_clips,
                            const int32_t* pair_clip, const int32_t* pair_delay, int32_t n_pairs, const double* partials) {
  VND_REQUIRE(rows >= 0 && n_clips >= 0 && n_pairs >= 0, VND_EINVAL, "negative extent (rows %lld, n_clips %d, n_pairs %d)", (long long)rows,
              n_clips, n_pairs);
  VND_REQUIRE(chan_stride >= rows, VND_EINVAL, "chan_stride %lld is shorter than rows = %lld: the two channels overlap", (long long)chan_stride,
              (long long)rows);
  if (n_pairs == 0) return VND_OK;
  VND_REQUIRE(n_clips > 0, VND_EINVAL, "%d pairs but no clips", n_pairs);
  VND_REQUIRE(x != nullptr || rows == 0, VND_EINVAL, "x is null");
  VND_REQUIRE(frame_offsets != nullptr && pair_clip != nullptr && pair_delay != nullptr && partials != nullptr, VND_EINVAL,
              "frame_offsets, pair_clip, pair_delay or partials is null");
  return VND_OK;
}

extern "C" int vnd_haas_objective_pairs_dev(const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets, int32_t n_clips,
                                            const int32_t* pair_clip, const int32_t* pair_delay, int32_t n_pairs, double* partials, void* stream) {
  int rc;
  if ((rc = check_haas_pairs(x, rows, chan_stride, frame_offsets, n_clips, pair_clip, pair_delay, n_pairs, partials))) return rc;
  return haas_objective_pairs_launch(x, chan_stride, reinterpret_cast<const long long*>(frame_offsets), pair_clip, pair_delay, n_pairs, partials,
                                     (cudaStream_t)stream);
}

// The clip and the candidate records of the one-clip family objectives: a float32 channel-planar clip of at least one frame.
static int check_family_clip(const float* x, int64_t frames, int64_t chan_stride, const void* cands, int32_t n_cand, const double* partials) {
  VND_REQUIRE(n_cand >= 0, VND_EINVAL, "negative n_cand %d", n_cand);
  // the reference takes max(|theta|) of the frames: an empty signal is a ValueError there (optimization.py:41-43)
  VND_REQUIRE(frames > 0, VND_EINVAL, "objective of an empty signal (zero-size array to reduction operation maximum which has no identity)");
  VND_REQUIRE(chan_stride >= frames, VND_EINVAL, "chan_stride %lld is shorter than frames = %lld: the two channels overlap", (long long)chan_stride,
              (long long)frames);
  VND_REQUIRE((x != nullptr && partials != nullptr) || n_cand == 0, VND_EINVAL, "x or partials is null");
  VND_REQUIRE(cands != nullptr || n_cand == 0, VND_EINVAL, "cands is null");
  return VND_OK;
}

static int check_vn_stereo(const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps, const vnd_vn_stereo_cand* cands,
                           int32_t n_cand, const double* partials) {
  int rc;
  if ((rc = check_family_clip(x, frames, chan_stride, cands, n_cand, partials)) || (rc = check_taps(taps))) return rc;
  VND_REQUIRE(taps->order == VND_ORDER_SEGMENTED, VND_EINVAL, "objective candidates need SEGMENTED tap programs");
  VND_REQUIRE((long long)taps->channels == 2LL * n_cand, VND_EINVAL, "the tap program has %d channels, %d candidates need %lld", taps->channels,
              n_cand, 2LL * n_cand);
  return VND_OK;
}

extern "C" int vnd_vn_stereo_objective_workspace(int64_t frames, int32_t n_cand, size_t* bytes) {
  VND_REQUIRE(bytes != nullptr, VND_EINVAL, "bytes is null");
  VND_REQUIRE(frames >= 0 && n_cand >= 0, VND_EINVAL, "negative extent");
  return vn_stereo_objective_workspace_bytes(frames, n_cand, bytes);
}

extern "C" int vnd_vn_stereo_objective_dev(const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps,
                                           const vnd_vn_stereo_cand* cands, int32_t n_cand, double* partials, void* workspace,
                                           size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_vn_stereo(x, frames, chan_stride, taps, cands, n_cand, partials))) return rc;
  return vn_stereo_objective_launch(x, frames, chan_stride, taps, cands, n_cand, partials, workspace, workspace_bytes, (cudaStream_t)stream);
}

static int check_vn_stereo_rms(const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps, const vnd_vn_stereo_cand* cands,
                               int32_t n_cand, const float* gains, const double* partials) {
  int rc;
  if ((rc = check_vn_stereo(x, frames, chan_stride, taps, cands, n_cand, partials))) return rc;
  VND_REQUIRE(gains != nullptr || n_cand == 0, VND_EINVAL, "gains is null");
  return VND_OK;
}

extern "C" int vnd_vn_stereo_rms_objective_workspace(int64_t frames, int32_t n_cand, size_t* bytes) {
  return vnd_vn_stereo_objective_workspace(frames, n_cand, bytes);
}

extern "C" int vnd_vn_stereo_rms_objective_dev(const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps,
                                               const vnd_vn_stereo_cand* cands, int32_t n_cand, float* gains, double* partials, void* workspace,
                                               size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_vn_stereo_rms(x, frames, chan_stride, taps, cands, n_cand, gains, partials))) return rc;
  return vn_stereo_rms_objective_launch(x, frames, chan_stride, taps, cands, n_cand, gains, partials, workspace, workspace_bytes,
                                        (cudaStream_t)stream);
}

extern "C" int vnd_haas_effect_objective_dev(const float* x, int64_t frames, int64_t chan_stride, const vnd_haas_clip* cands, int32_t n_cand,
                                             double* partials, void* stream) {
  int rc;
  if ((rc = check_family_clip(x, frames, chan_stride, cands, n_cand, partials))) return rc;
  VND_REQUIRE(reinterpret_cast<uintptr_t>(cands) % 16 == 0, VND_EINVAL, "cands must be 16-byte aligned");
  return haas_effect_objective_launch(x, frames, chan_stride, cands, n_cand, partials, (cudaStream_t)stream);
}

// Host frame offsets of n clips (n + 1 values): from 0, never decreasing, ending at rows.
static int check_offsets(const int64_t* offs, int32_t n, int64_t rows) {
  VND_REQUIRE(offs[0] == 0, VND_EINVAL, "frame_offsets[0] is %lld, not 0", (long long)offs[0]);
  for (int i = 0; i < n; ++i)
    VND_REQUIRE(offs[i + 1] >= offs[i], VND_EINVAL, "frame_offsets decrease at clip %d (%lld -> %lld)", i, (long long)offs[i],
                (long long)offs[i + 1]);
  VND_REQUIRE(offs[n] == rows, VND_EINVAL, "frame_offsets end at %lld, not at rows = %lld", (long long)offs[n], (long long)rows);
  return VND_OK;
}

// Host tables of the run-list objective: offsets (check_offsets) and every run's clip.  Runs of at least one candidate
// need a clip with frames.
static int check_run_clips(int64_t rows, const int64_t* offs, int32_t n_clips, const int32_t* run_clip, const int32_t* run_count, int32_t n_runs) {
  VND_REQUIRE(rows >= 0 && n_clips >= 0 && n_runs >= 0, VND_EINVAL, "negative extent (rows %lld, n_clips %d, n_runs %d)", (long long)rows,
              n_clips, n_runs);
  VND_REQUIRE(offs != nullptr, VND_EINVAL, "frame_offsets is null");
  int rc;
  if ((rc = check_offsets(offs, n_clips, rows))) return rc;
  if (n_runs == 0) return VND_OK;
  VND_REQUIRE(run_clip != nullptr && run_count != nullptr, VND_EINVAL, "run_clip or run_count is null");
  for (int r = 0; r < n_runs; ++r) {
    const int c = run_clip[r];
    VND_REQUIRE(c >= 0 && c < n_clips, VND_EINVAL, "run_clip[%d] = %d is outside [0, %d)", r, c, n_clips);
    VND_REQUIRE(run_count[r] >= 0, VND_EINVAL, "run_count[%d] = %d is negative", r, run_count[r]);
    // the reference takes max(|theta|) of the frames: an empty signal is a ValueError there (optimization.py:41-43)
    VND_REQUIRE(run_count[r] == 0 || offs[c + 1] > offs[c], VND_EINVAL,
                "run %d: objective of an empty signal (clip %d has no frames: zero-size array to reduction operation maximum which has no identity)",
                r, c);
  }
  return VND_OK;
}

// Everything vnd_vn_objective_runs_dev can check on the host before it touches the device.
static int check_runs(const float* x, int64_t rows, int64_t chan_stride, const int64_t* offs, int32_t n_clips, const vnd_tap_program* cand,
                      const int32_t* run_clip, const int32_t* run_cand, const int32_t* run_count, const int32_t* run_out, int32_t n_runs,
                      const double* partials, int64_t n_partial_rows) {
  int rc;
  if ((rc = check_taps(cand))) return rc;
  VND_REQUIRE(cand->order == VND_ORDER_SEGMENTED, VND_EINVAL, "objective candidates need SEGMENTED tap programs");
  VND_REQUIRE(chan_stride >= rows, VND_EINVAL, "chan_stride %lld is shorter than rows = %lld: the two channels overlap", (long long)chan_stride,
              (long long)rows);
  VND_REQUIRE(n_partial_rows >= 0, VND_EINVAL, "negative n_partial_rows %lld", (long long)n_partial_rows);
  if ((rc = check_run_clips(rows, offs, n_clips, run_clip, run_count, n_runs))) return rc;
  if (n_runs == 0) return VND_OK;
  VND_REQUIRE(run_cand != nullptr && run_out != nullptr, VND_EINVAL, "run_cand or run_out is null");
  for (int r = 0; r < n_runs; ++r) {
    VND_REQUIRE(run_cand[r] >= 0 && (long long)run_cand[r] + run_count[r] <= cand->channels, VND_EINVAL,
                "run %d: channels [%d, %lld) are outside the program's %d", r, run_cand[r], (long long)run_cand[r] + run_count[r], cand->channels);
    VND_REQUIRE(run_out[r] >= 0 && (long long)run_out[r] + run_count[r] <= n_partial_rows, VND_EINVAL,
                "run %d: output rows [%d, %lld) are outside the %lld partial rows", r, run_out[r], (long long)run_out[r] + run_count[r],
                (long long)n_partial_rows);
  }
  VND_REQUIRE(x != nullptr || rows == 0, VND_EINVAL, "x is null");
  VND_REQUIRE(partials != nullptr || n_partial_rows == 0, VND_EINVAL, "partials is null");
  return VND_OK;
}

extern "C" int vnd_vn_objective_runs_workspace(const int64_t* frame_offsets, int32_t n_clips, const int32_t* run_clip, const int32_t* run_count,
                                               int32_t n_runs, size_t* bytes) {
  VND_REQUIRE(bytes != nullptr, VND_EINVAL, "bytes is null");
  VND_REQUIRE(frame_offsets != nullptr && n_clips >= 0, VND_EINVAL, "frame_offsets is null or n_clips negative");
  int rc;
  if ((rc = check_run_clips(frame_offsets[n_clips], frame_offsets, n_clips, run_clip, run_count, n_runs))) return rc;
  if (n_runs == 0) {
    *bytes = 0;
    return VND_OK;
  }
  return objective_runs_workspace_bytes(reinterpret_cast<const long long*>(frame_offsets), run_clip, run_count, n_runs, bytes);
}

extern "C" int vnd_vn_objective_runs_dev(const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets, int32_t n_clips,
                                         const vnd_tap_program* cand, const int32_t* run_clip, const int32_t* run_cand, const int32_t* run_count,
                                         const int32_t* run_out, int32_t n_runs, double* partials, int64_t n_partial_rows, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_runs(x, rows, chan_stride, frame_offsets, n_clips, cand, run_clip, run_cand, run_count, run_out, n_runs, partials,
                       n_partial_rows)))
    return rc;
  if (n_runs == 0) return VND_OK;
  return vn_objective_runs_launch(x, chan_stride, reinterpret_cast<const long long*>(frame_offsets), run_clip, run_cand, run_count, run_out, n_runs,
                                  cand, partials, workspace, workspace_bytes, (cudaStream_t)stream);
}

static int check_flat(const vnd_signal* s, int ndim, const char* name) {
  int rc;
  if ((rc = check_signal(s, name))) return rc;
  VND_REQUIRE(ndim == 1 || ndim == 2, VND_EINVAL, "%s: ndim must be 1 or 2", name);
  if (ndim == 1) VND_REQUIRE(s->stride_t == 1 || s->frames <= 1, VND_EUNSUPPORTED, "%s must be contiguous", name);
  else VND_REQUIRE((s->stride_c == 1 || s->channels <= 1) && (s->stride_t == s->channels || s->frames <= 1), VND_EUNSUPPORTED,
                   "%s must be a contiguous C-order (frames, channels) array", name);
  return VND_OK;
}

extern "C" int vnd_dsp_workspace(int64_t elems, size_t* bytes) {
  VND_REQUIRE(bytes != nullptr && elems >= 0, VND_EINVAL, "bad argument");
  *bytes = dsp_workspace_bytes(elems);
  return VND_OK;
}

static int check_rms_normalize(const vnd_signal* x, int32_t x_ndim, const vnd_signal* y, int32_t y_ndim) {
  int rc;
  if ((rc = check_flat(x, x_ndim, "input_signal")) || (rc = check_flat(y, y_ndim, "output_signal"))) return rc;
  VND_REQUIRE(x->dtype == y->dtype, VND_EINVAL, "input and output must have the same dtype");
  return VND_OK;
}

extern "C" int vnd_rms_normalize_dev(const vnd_signal* x, int32_t x_ndim, const vnd_signal* y, int32_t y_ndim, int32_t stereo_mode, double epsilon,
                                     void* workspace, size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_rms_normalize(x, x_ndim, y, y_ndim))) return rc;
  const long long nx = x->frames * (long long)(x_ndim == 1 ? 1 : x->channels), ny = y->frames * (long long)(y_ndim == 1 ? 1 : y->channels);
  VND_REQUIRE(workspace != nullptr && workspace_bytes >= dsp_workspace_bytes(nx > ny ? nx : ny), VND_ENOMEM, "dsp workspace too small");
  return rms_normalize_launch(x, y, x_ndim, y_ndim, stereo_mode, epsilon, workspace, (cudaStream_t)stream);
}

extern "C" int vnd_peak_normalize_dev(const vnd_signal* y, int32_t ndim, int32_t stereo_mode, double epsilon, void* workspace, size_t workspace_bytes,
                                      void* stream) {
  int rc;
  if ((rc = check_flat(y, ndim, "input_signal"))) return rc;
  VND_REQUIRE(workspace != nullptr && workspace_bytes >= dsp_workspace_bytes(0), VND_ENOMEM, "dsp workspace too small");
  return peak_normalize_launch(y, ndim, stereo_mode, epsilon, workspace, (cudaStream_t)stream);
}

static int check_polar(const void* left, const void* right, int64_t n, int32_t dtype, const void* radii, const void* thetas) {
  VND_REQUIRE(n >= 0, VND_EINVAL, "negative length");
  VND_REQUIRE(dtype == VND_F32 || dtype == VND_F64, VND_EINVAL, "unknown dtype %d", dtype);
  VND_REQUIRE(n == 0 || (left && right && radii && thetas), VND_EINVAL, "null buffer");
  return VND_OK;
}

extern "C" int vnd_polar_dev(const void* left, const void* right, int64_t n, int32_t dtype, int32_t mode_ms, int32_t semicircular, int32_t normalize,
                             void* radii, void* thetas, void* weights, void* workspace, size_t workspace_bytes, void* stream) {
  int rc;
  if ((rc = check_polar(left, right, n, dtype, radii, thetas))) return rc;
  VND_REQUIRE(workspace != nullptr && workspace_bytes >= dsp_workspace_bytes(n), VND_ENOMEM, "dsp workspace too small");
  return polar_launch(left, right, n, dtype, mode_ms, semicircular, normalize, radii, thetas, weights, workspace, (cudaStream_t)stream);
}

// ================================================================================================
// host entry points
// ================================================================================================
struct vnd_ctx {
  int device = 0;
  cudaStream_t streams[3] = {nullptr, nullptr, nullptr};
  struct Buf {
    void* p = nullptr;
    size_t cap = 0;
  };
  Buf slots[18];  // grow-only device arena
  Buf pin[4];     // grow-only page-locked staging for pageable callers: [0,1] upload ring, [2,3] download ring
  std::mutex mu;
};

namespace {

enum Slot { S_IN = 0, S_OUT = 1, S_WORK = 2, S_WORDS = 3, S_OFFS = 4, S_AUX = 5, S_RING = 6 /* 6..11 */, S_SCRATCH = 12 /* 12..17 */ };

int arena(vnd_ctx* ctx, int slot, size_t bytes, void** out) {
  vnd_ctx::Buf& b = ctx->slots[slot];
  if (bytes == 0) bytes = 16;
  if (b.cap < bytes) {
    if (b.p) VND_CUDA_OK(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    const size_t want = align_up(bytes + bytes / 8, 1 << 20);
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      set_error("device arena: cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
      return VND_ENOMEM;
    }
    b.cap = want;
  }
  *out = b.p;
  return VND_OK;
}

// A strided host view is "dense" when it covers one contiguous block: C-order (frames, channels),
// planar (channels, frames), or a mono signal broadcast with stride_c == 0.
struct Dense {
  size_t elems;
  bool ok;
};
Dense dense_extent(const vnd_signal* s) {
  const long long L = s->frames, C = s->channels;
  if (L * C == 0) return {0, true};
  if (s->stride_c == 0 && s->stride_t == 1) return {(size_t)L, true};
  if (C == 1 && s->stride_t == 1) return {(size_t)L, true};
  if (s->stride_c == 1 && s->stride_t == C) return {(size_t)(L * C), true};
  if (s->stride_t == 1 && s->stride_c == L) return {(size_t)(L * C), true};
  return {0, false};
}

size_t esize(int dtype) { return dtype == VND_F64 ? 8 : 4; }

// Arena slot `slot`, holding a copy of `bytes` host bytes from `src` once stream `st` gets there.
int upload(vnd_ctx* ctx, int slot, const void* src, size_t bytes, cudaStream_t st, void** dev) {
  int rc;
  if ((rc = arena(ctx, slot, bytes, dev))) return rc;
  if (bytes) VND_CUDA_OK(cudaMemcpyAsync(*dev, src, bytes, cudaMemcpyHostToDevice, st));
  return VND_OK;
}

int upload_program(vnd_ctx* ctx, const vnd_tap_program* host, vnd_tap_program* dev, cudaStream_t st) {
  *dev = *host;
  void *w = nullptr, *o = nullptr;
  int rc;
  if ((rc = upload(ctx, S_WORDS, host->words, (size_t)host->n_words * 4, st, &w)) ||
      (rc = upload(ctx, S_OFFS, host->offsets, host->channels ? ((size_t)host->channels + 1) * 4 : 0, st, &o)))
    return rc;
  dev->words = reinterpret_cast<const int32_t*>(w);
  dev->offsets = reinterpret_cast<const int32_t*>(o);
  return VND_OK;
}

// Does the calling thread have a CUDA context bound?  (cudaGetDevice answers 0 either way, and since CUDA 12
// cudaSetDevice CREATES the primary context of the device it names.)
bool thread_has_context() {
  typedef CUresult (*GetCurrentFn)(CUcontext*);
  static GetCurrentFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuCtxGetCurrent", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
    (void)cudaGetLastError();
    return reinterpret_cast<GetCurrentFn>(p);
  }();
  if (!fn) return true;  // cannot tell: behave like a plain save / restore
  CUcontext c = nullptr;
  return fn(&c) == CUDA_SUCCESS && c != nullptr;
}

// Selects the context's device for the duration of a call.  The previous device is restored only if the thread
// HAD a context before: restoring "device 0" for a thread that never touched CUDA would create a primary context
// (about half a GB) on GPU 0 in every rank of a multi-GPU job, and fails under exclusive-process compute mode.
struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (thread_has_context()) {
      if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    }
    ok = (prev == dev) || cudaSetDevice(dev) == cudaSuccess;
    if (prev == dev) prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

#define VND_ENTER(ctx)                                                      \
  VND_REQUIRE((ctx) != nullptr, VND_EINVAL, "context is null");             \
  std::lock_guard<std::mutex> _lock((ctx)->mu);                             \
  DeviceGuard _guard((ctx)->device);                                        \
  VND_REQUIRE(_guard.ok, VND_ECUDA, "cudaSetDevice(%d) failed", (ctx)->device)

}  // namespace

extern "C" int vnd_ctx_create(int device, vnd_ctx** out) {
  VND_REQUIRE(out != nullptr, VND_EINVAL, "ctx out pointer is null");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    (void)cudaGetLastError();
    set_error("no CUDA device available (%s); this library has no CPU fallback", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    return VND_ECUDA;
  }
  VND_REQUIRE(device >= 0 && device < n, VND_EINVAL, "device %d out of range (have %d)", device, n);
  vnd_ctx* ctx = new vnd_ctx();
  ctx->device = device;
  DeviceGuard guard(device);
  for (auto& s : ctx->streams) {
    if (cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking) != cudaSuccess) {
      set_error("cudaStreamCreate failed");
      delete ctx;
      return VND_ECUDA;
    }
  }
  *out = ctx;
  return VND_OK;
}

extern "C" int vnd_ctx_destroy(vnd_ctx* ctx) {
  if (!ctx) return VND_OK;
  {
    DeviceGuard guard(ctx->device);
    for (auto& s : ctx->streams)
      if (s) {
        cudaStreamSynchronize(s);
        cudaStreamDestroy(s);
      }
    for (auto& b : ctx->slots)
      if (b.p) cudaFree(b.p);
    for (auto& b : ctx->pin)
      if (b.p) cudaFreeHost(b.p);
  }
  delete ctx;
  return VND_OK;
}

extern "C" int vnd_host_alloc(size_t bytes, void** ptr) {
  VND_REQUIRE(ptr != nullptr, VND_EINVAL, "ptr is null");
  *ptr = nullptr;
  VND_CUDA_OK(cudaHostAlloc(ptr, bytes ? bytes : 16, cudaHostAllocPortable));
  return VND_OK;
}

extern "C" int vnd_ctx_host_alloc(vnd_ctx* ctx, size_t bytes, void** ptr) {
  VND_REQUIRE(ctx != nullptr, VND_EINVAL, "context is null");
  VND_REQUIRE(ptr != nullptr, VND_EINVAL, "ptr is null");
  *ptr = nullptr;
  DeviceGuard guard(ctx->device);
  VND_REQUIRE(guard.ok, VND_ECUDA, "cudaSetDevice(%d) failed", ctx->device);
  VND_CUDA_OK(cudaHostAlloc(ptr, bytes ? bytes : 16, cudaHostAllocPortable));
  return VND_OK;
}

extern "C" int vnd_host_free(void* ptr) {
  if (ptr) VND_CUDA_OK(cudaFreeHost(ptr));
  return VND_OK;
}

extern "C" int vnd_rms_normalize_host(vnd_ctx* ctx, const vnd_signal* x, int32_t x_ndim, const vnd_signal* y, int32_t y_ndim, int32_t stereo_mode,
                                      double epsilon) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_rms_normalize(x, x_ndim, y, y_ndim))) return rc;
  const size_t es = esize(x->dtype);
  const size_t nx = (size_t)x->frames * (x_ndim == 1 ? 1 : x->channels), ny = (size_t)y->frames * (y_ndim == 1 ? 1 : y->channels);
  cudaStream_t st = ctx->streams[0];
  void *dx = nullptr, *dy = nullptr, *work = nullptr;
  const size_t wbytes = dsp_workspace_bytes((long long)(nx > ny ? nx : ny));
  if ((rc = upload(ctx, S_IN, x->data, nx * es, st, &dx)) || (rc = upload(ctx, S_OUT, y->data, ny * es, st, &dy)) ||
      (rc = arena(ctx, S_WORK, wbytes, &work)))
    return rc;
  vnd_signal xd = *x, yd = *y;
  xd.data = dx;
  yd.data = dy;
  if ((rc = vnd_rms_normalize_dev(&xd, x_ndim, &yd, y_ndim, stereo_mode, epsilon, work, wbytes, st))) return rc;
  if (ny) VND_CUDA_OK(cudaMemcpyAsync(y->data, dy, ny * es, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_peak_normalize_host(vnd_ctx* ctx, const vnd_signal* y, int32_t ndim, int32_t stereo_mode, double epsilon) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_flat(y, ndim, "input_signal"))) return rc;
  const size_t es = esize(y->dtype), ny = (size_t)y->frames * (ndim == 1 ? 1 : y->channels);
  cudaStream_t st = ctx->streams[0];
  void *dy = nullptr, *work = nullptr;
  const size_t wbytes = dsp_workspace_bytes(0);
  if ((rc = upload(ctx, S_IN, y->data, ny * es, st, &dy)) || (rc = arena(ctx, S_WORK, wbytes, &work))) return rc;
  vnd_signal yd = *y;
  yd.data = dy;
  if ((rc = vnd_peak_normalize_dev(&yd, ndim, stereo_mode, epsilon, work, wbytes, st))) return rc;
  if (ny) VND_CUDA_OK(cudaMemcpyAsync(y->data, dy, ny * es, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_polar_host(vnd_ctx* ctx, const void* left, const void* right, int64_t n, int32_t dtype, int32_t mode_ms, int32_t semicircular,
                              int32_t normalize, void* radii, void* thetas, void* weights) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_polar(left, right, n, dtype, radii, thetas))) return rc;
  if (n == 0) return VND_OK;
  const size_t bytes = (size_t)n * esize(dtype);
  cudaStream_t st = ctx->streams[0];
  void *din = nullptr, *dout = nullptr, *work = nullptr;
  const size_t wbytes = dsp_workspace_bytes(n);
  if ((rc = arena(ctx, S_IN, 2 * bytes, &din)) || (rc = arena(ctx, S_OUT, 3 * bytes, &dout)) || (rc = arena(ctx, S_WORK, wbytes, &work))) return rc;
  char *dl = (char*)din, *dr = dl + bytes, *drad = (char*)dout, *dth = drad + bytes, *dw = dth + bytes;
  VND_CUDA_OK(cudaMemcpyAsync(dl, left, bytes, cudaMemcpyHostToDevice, st));
  VND_CUDA_OK(cudaMemcpyAsync(dr, right, bytes, cudaMemcpyHostToDevice, st));
  if ((rc = vnd_polar_dev(dl, dr, n, dtype, mode_ms, semicircular, normalize, drad, dth, weights ? dw : nullptr, work, wbytes, st))) return rc;
  VND_CUDA_OK(cudaMemcpyAsync(radii, drad, bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaMemcpyAsync(thetas, dth, bytes, cudaMemcpyDeviceToHost, st));
  if (weights) VND_CUDA_OK(cudaMemcpyAsync(weights, dw, bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

// ================================================================================================
// overlapped host path: upload / kernels / download of consecutive chunks on three streams
// ================================================================================================
namespace {

int staging(vnd_ctx* ctx, int slot, size_t bytes, void** out) {
  vnd_ctx::Buf& b = ctx->pin[slot];
  if (b.cap < bytes) {
    if (b.p) VND_CUDA_OK(cudaFreeHost(b.p));
    b.p = nullptr;
    b.cap = 0;
    cudaError_t e = cudaHostAlloc(&b.p, bytes, cudaHostAllocDefault);
    if (e != cudaSuccess) {
      (void)cudaGetLastError();
      set_error("pinned staging: cudaHostAlloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
      return VND_ENOMEM;
    }
    b.cap = bytes;
  }
  *out = b.p;
  return VND_OK;
}

// Page-locked (cudaHostAlloc / cudaHostRegister) memory is copied by DMA straight from / to the caller's
// buffer; anything else goes through the context's staging ring.
bool is_page_locked(const void* p) {
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    (void)cudaGetLastError();
    return false;
  }
  return a.type == cudaMemoryTypeHost;
}

struct PipeChunk {
  const char* src;   // host bytes uploaded for this chunk (contiguous)
  size_t src_bytes;
  char* dst;         // host bytes this chunk produces (contiguous)
  size_t dst_bytes;
};

struct PipeSync {
  std::mutex mu;
  std::condition_variable cv;
  long long staged = -1, h2d_enqueued = -1, d2h_enqueued = -1, copied = -1;
  bool abort = false;
  void set(long long PipeSync::*field, long long v) {
    {
      std::lock_guard<std::mutex> l(mu);
      this->*field = v;
    }
    cv.notify_all();
  }
  bool wait(long long PipeSync::*field, long long v) {  // false when the pipeline was aborted
    std::unique_lock<std::mutex> l(mu);
    cv.wait(l, [&] { return abort || this->*field >= v; });
    return !abort;
  }
  void stop() {
    {
      std::lock_guard<std::mutex> l(mu);
      abort = true;
    }
    cv.notify_all();
  }
};

constexpr int kPipeSlots = 3;

// Runs n chunks through a ring of kPipeSlots device buffers: ctx->streams[0] uploads, [1] computes, [2] downloads,
// ordered by events, so the upload of chunk k + 1 and the download of chunk k - 1 overlap the kernels of chunk k
// (PCIe is full duplex).  `compute(k, din, dout, scratch_a, scratch_b, stream)` enqueues the kernels of chunk k.
// Pageable host buffers are staged through the context's page-locked ring by two helper threads (one copies
// chunks in ahead of the uploads, one copies finished chunks out), so the caller's thread only enqueues.
template <class ChunkOf, class Compute>
int run_pipeline(vnd_ctx* ctx, int n, size_t in_cap, size_t out_cap, size_t scratch_cap, ChunkOf chunk_of, Compute compute) {
  if (n <= 0) return VND_OK;
  int rc;
  cudaStream_t up = ctx->streams[0], comp = ctx->streams[1], down = ctx->streams[2];
  void *din[kPipeSlots], *dout[kPipeSlots], *sa[kPipeSlots], *sb[kPipeSlots];
  for (int s = 0; s < kPipeSlots; ++s) {
    if ((rc = arena(ctx, S_RING + 2 * s, in_cap, &din[s]))) return rc;
    if ((rc = arena(ctx, S_RING + 2 * s + 1, out_cap, &dout[s]))) return rc;
    sa[s] = sb[s] = nullptr;
    if (scratch_cap) {
      if ((rc = arena(ctx, S_SCRATCH + 2 * s, scratch_cap, &sa[s]))) return rc;
      if ((rc = arena(ctx, S_SCRATCH + 2 * s + 1, scratch_cap, &sb[s]))) return rc;
    }
  }
  const PipeChunk first = chunk_of(0);
  const bool in_locked = is_page_locked(first.src), out_locked = is_page_locked(first.dst);
  void *pin_in[2] = {nullptr, nullptr}, *pin_out[2] = {nullptr, nullptr};
  if (!in_locked)
    for (int i = 0; i < 2; ++i)
      if ((rc = staging(ctx, i, in_cap, &pin_in[i]))) return rc;
  if (!out_locked)
    for (int i = 0; i < 2; ++i)
      if ((rc = staging(ctx, 2 + i, out_cap, &pin_out[i]))) return rc;

  std::vector<cudaEvent_t> ev(3 * (size_t)n, nullptr);
  auto ev_up = [&](int k) -> cudaEvent_t& { return ev[3 * (size_t)k]; };
  auto ev_comp = [&](int k) -> cudaEvent_t& { return ev[3 * (size_t)k + 1]; };
  auto ev_down = [&](int k) -> cudaEvent_t& { return ev[3 * (size_t)k + 2]; };
  rc = VND_OK;
  for (auto& e : ev)
    if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) {
      set_error("cudaEventCreate failed");
      rc = VND_ECUDA;
      break;
    }

  PipeSync sync;
  std::thread stage_in, stage_out;
  const int device = ctx->device;
  if (rc == VND_OK && !in_locked)
    stage_in = std::thread([&] {  // copies chunk k into staging slot k % 2 once the upload of chunk k - 2 has left it
      cudaSetDevice(device);
      for (int k = 0; k < n; ++k) {
        if (k >= 2) {
          if (!sync.wait(&PipeSync::h2d_enqueued, k - 2)) return;
          if (cudaEventSynchronize(ev_up(k - 2)) != cudaSuccess) return sync.stop();
        }
        const PipeChunk c = chunk_of(k);
        memcpy(pin_in[k & 1], c.src, c.src_bytes);
        sync.set(&PipeSync::staged, k);
      }
    });
  if (rc == VND_OK && !out_locked)
    stage_out = std::thread([&] {  // copies finished chunk k out of staging slot k % 2
      cudaSetDevice(device);
      for (int k = 0; k < n; ++k) {
        if (!sync.wait(&PipeSync::d2h_enqueued, k)) return;
        if (cudaEventSynchronize(ev_down(k)) != cudaSuccess) return sync.stop();
        const PipeChunk c = chunk_of(k);
        memcpy(c.dst, pin_out[k & 1], c.dst_bytes);
        sync.set(&PipeSync::copied, k);
      }
    });

#define VND_PIPE_OK(expr)                                                                           \
  if (rc == VND_OK) {                                                                               \
    cudaError_t _e = (expr);                                                                        \
    if (_e != cudaSuccess) {                                                                        \
      set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__);        \
      rc = VND_ECUDA;                                                                               \
    }                                                                                               \
  }
  for (int k = 0; k < n && rc == VND_OK; ++k) {
    const int s = k % kPipeSlots;
    const PipeChunk c = chunk_of(k);
    // upload (the slot's input buffer is free once the kernels of chunk k - slots have run)
    if (k >= kPipeSlots) VND_PIPE_OK(cudaStreamWaitEvent(up, ev_comp(k - kPipeSlots), 0));
    if (!in_locked && !sync.wait(&PipeSync::staged, k)) {
      set_error("pipeline staging failed");
      rc = VND_ECUDA;
      break;
    }
    VND_PIPE_OK(cudaMemcpyAsync(din[s], in_locked ? (const void*)c.src : pin_in[k & 1], c.src_bytes, cudaMemcpyHostToDevice, up));
    VND_PIPE_OK(cudaEventRecord(ev_up(k), up));
    if (!in_locked) sync.set(&PipeSync::h2d_enqueued, k);
    // kernels (the slot's output buffer is free once chunk k - slots has been downloaded)
    VND_PIPE_OK(cudaStreamWaitEvent(comp, ev_up(k), 0));
    if (k >= kPipeSlots) VND_PIPE_OK(cudaStreamWaitEvent(comp, ev_down(k - kPipeSlots), 0));
    if (rc == VND_OK) rc = compute(k, din[s], dout[s], sa[s], sb[s], comp);
    VND_PIPE_OK(cudaEventRecord(ev_comp(k), comp));
    // download
    VND_PIPE_OK(cudaStreamWaitEvent(down, ev_comp(k), 0));
    if (!out_locked && k >= 2 && !sync.wait(&PipeSync::copied, k - 2)) {
      set_error("pipeline staging failed");
      rc = VND_ECUDA;
      break;
    }
    VND_PIPE_OK(cudaMemcpyAsync(out_locked ? (void*)c.dst : pin_out[k & 1], dout[s], c.dst_bytes, cudaMemcpyDeviceToHost, down));
    VND_PIPE_OK(cudaEventRecord(ev_down(k), down));
    if (!out_locked && rc == VND_OK) sync.set(&PipeSync::d2h_enqueued, k);
  }
  if (rc != VND_OK) sync.stop();
  if (stage_in.joinable()) stage_in.join();
  if (stage_out.joinable()) stage_out.join();
  for (auto& st : ctx->streams) {
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess && rc == VND_OK) {
      set_error("cudaStreamSynchronize failed: %s", cudaGetErrorString(e));
      rc = VND_ECUDA;
    }
  }
  if (rc == VND_OK && sync.abort) {
    set_error("pipeline staging thread failed");
    rc = VND_ECUDA;
  }
  for (auto& e : ev)
    if (e) cudaEventDestroy(e);
#undef VND_PIPE_OK
  return rc;
}

size_t pipe_chunk_bytes() {  // bytes uploaded per pipeline stage (VND_PIPE_CHUNK_MB, default 64)
  const char* e = getenv("VND_PIPE_CHUNK_MB");
  const long mb = e ? atol(e) : 64;
  return (size_t)(mb > 0 ? mb : 64) << 20;
}
constexpr size_t kPipeMinBytes = 8u << 20;  // below this one blocking copy each way is as fast

// Does an upload of `in_bytes` go through run_pipeline?  VND_NO_PIPELINE forces the one-shot path, the reference
// the pipelined one is tested against.
bool pipelined(size_t in_bytes) { return in_bytes >= kPipeMinBytes && getenv("VND_NO_PIPELINE") == nullptr; }

// Chunks of whole clips of a packed (rows, 2) float32 batch of about pipe_chunk_bytes() each (at least four chunks when
// there are four clips): first[k] .. first[k + 1] are the clips of chunk k.
std::vector<int> clip_chunks(const int64_t* offs, int32_t n_clips, int64_t rows) {
  size_t target = pipe_chunk_bytes();
  if (target > (size_t)rows * 8 / 4) target = (size_t)rows * 8 / 4;
  std::vector<int> first{0};
  while (first.back() < n_clips) {
    const int a = first.back();
    int b = a + 1;
    while (b < n_clips && (size_t)(offs[b + 1] - offs[a]) * 8 <= target) ++b;
    first.push_back(b);
  }
  return first;
}

// Planar (channels, frames) float32 host slabs: chunks are groups of whole channels.
int fir_pipeline_planar(vnd_ctx* ctx, const float* x, float* y, long long frames, int channels, const vnd_tap_program* dprog,
                        int channels_per_chunk) {
  if (channels_per_chunk <= 0) {
    long long cpc = (long long)(pipe_chunk_bytes() / ((size_t)frames * 4));
    if (cpc > (channels + 3) / 4) cpc = (channels + 3) / 4;  // at least four stages when there are four channels
    channels_per_chunk = (int)(cpc < 1 ? 1 : cpc);
  }
  if (channels_per_chunk > channels) channels_per_chunk = channels;
  const int n = (channels + channels_per_chunk - 1) / channels_per_chunk;
  const size_t cap = (size_t)channels_per_chunk * frames * 4;
  auto chunk_of = [&](int k) {
    const int c0 = k * channels_per_chunk;
    const int nc = channels - c0 < channels_per_chunk ? channels - c0 : channels_per_chunk;
    const size_t bytes = (size_t)nc * frames * 4;
    return PipeChunk{reinterpret_cast<const char*>(x + (size_t)c0 * frames), bytes, reinterpret_cast<char*>(y + (size_t)c0 * frames), bytes};
  };
  auto compute = [&](int k, void* din, void* dout, void*, void*, cudaStream_t st) {
    const int c0 = k * channels_per_chunk;
    const int nc = channels - c0 < channels_per_chunk ? channels - c0 : channels_per_chunk;
    vnd_signal xd{din, frames, nc, VND_F32, 1, frames};
    vnd_signal yd{dout, frames, nc, VND_F32, 1, frames};
    vnd_tap_program sub = *dprog;
    sub.channels = nc;
    sub.offsets = dprog->offsets + c0;
    return vnd_sparse_fir_dev(&xd, &yd, &sub, st);
  };
  return run_pipeline(ctx, n, cap, cap, 0, chunk_of, compute);
}

// C-order (frames, channels) float32 host slabs - the reference's layout: chunks are runs of frames (all channels,
// contiguous on the host) uploaded with the filter's halo behind them; wide chunks are transposed to planar on the
// device around the planar kernel, so that tiles load and store coalesced.
int fir_pipeline_interleaved(vnd_ctx* ctx, const float* x, int x_channels, float* y, long long frames, int channels,
                             const vnd_tap_program* dprog) {
  long long halo = dprog->halo > 0 ? dprog->halo : 0;
  halo = (halo + 3) & ~3LL;
  long long T = (long long)(pipe_chunk_bytes() / ((size_t)x_channels * 4));
  if (T > (frames + 3) / 4) T = (frames + 3) / 4;
  if (T < 4 * halo) T = 4 * halo;  // the halo is uploaded twice: keep that below a quarter
  T = (T + 3) & ~3LL;
  if (T < 4) T = 4;
  const int n = (int)((frames + T - 1) / T);
  const bool wide = channels > 2 && x_channels == channels;
  const size_t in_cap = (size_t)(T + halo) * x_channels * 4, out_cap = (size_t)(T + halo) * channels * 4;
  auto span_of = [&](int k, long long* t0, long long* nt, long long* nin) {
    *t0 = (long long)k * T;
    *nt = frames - *t0 < T ? frames - *t0 : T;
    *nin = frames - *t0 < T + halo ? frames - *t0 : T + halo;  // frames uploaded: the chunk and its halo, clipped at the end
  };
  auto chunk_of = [&](int k) {
    long long t0, nt, nin;
    span_of(k, &t0, &nt, &nin);
    return PipeChunk{reinterpret_cast<const char*>(x + (size_t)t0 * x_channels), (size_t)nin * x_channels * 4,
                     reinterpret_cast<char*>(y + (size_t)t0 * channels), (size_t)nt * channels * 4};
  };
  auto compute = [&](int k, void* din, void* dout, void* sa, void* sb, cudaStream_t st) {
    long long t0, nt, nin;
    span_of(k, &t0, &nt, &nin);
    int rc;
    if (wide) {
      const long long ld = (nin + 3) & ~3LL;  // planar channel pitch: a multiple of 4 keeps the bulk-copy path
      if ((rc = transpose_launch_ld((const float*)din, (float*)sa, nin, channels, channels, ld, st))) return rc;
      vnd_signal xp{sa, nin, channels, VND_F32, 1, ld};
      vnd_signal yp{sb, nin, channels, VND_F32, 1, ld};
      if ((rc = vnd_sparse_fir_dev(&xp, &yp, dprog, st))) return rc;
      return transpose_launch_ld((const float*)sb, (float*)dout, channels, nt, ld, channels, st);
    }
    vnd_signal xd{din, nin, x_channels, VND_F32, x_channels, 1};
    vnd_signal yd{dout, nin, channels, VND_F32, channels, 1};
    return vnd_sparse_fir_dev(&xd, &yd, dprog, st);
  };
  return run_pipeline(ctx, n, in_cap, out_cap, wide ? (size_t)(T + halo + 4) * channels * 4 : 0, chunk_of, compute);
}

}  // namespace

extern "C" int vnd_sparse_fir_host(vnd_ctx* ctx, const vnd_signal* x, const vnd_signal* y, const vnd_tap_program* taps) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_sparse_fir(x, y, taps))) return rc;
  const Dense dx = dense_extent(x), dy = dense_extent(y);
  VND_REQUIRE(dx.ok && dy.ok, VND_EUNSUPPORTED, "host signals must be contiguous C-order (frames, channels) or planar (channels, frames)");
  cudaStream_t st = ctx->streams[0];
  vnd_tap_program dprog;
  if ((rc = upload_program(ctx, taps, &dprog, st))) return rc;
  // Large float32 slabs: upload, kernels and download overlapped chunk by chunk (run_pipeline)
  if (x->dtype == VND_F32 && x->stride_c != 0 && pipelined(dx.elems * 4)) {
    const long long L = x->frames;
    const int C = y->channels;
    const bool x_planar = x->stride_t == 1 && (x->stride_c == L || x->channels == 1), y_planar = y->stride_t == 1 && (y->stride_c == L || C == 1);
    const bool x_inter = x->stride_c == 1 && x->stride_t == x->channels, y_inter = y->stride_c == 1 && y->stride_t == C;
    VND_CUDA_OK(cudaStreamSynchronize(st));  // the program is on the device before the other streams read it
    if (x_planar && y_planar && x->channels == C && C > 1)
      return fir_pipeline_planar(ctx, (const float*)x->data, (float*)y->data, L, C, &dprog, 0);
    if (x_inter && y_inter && L >= 16LL * (taps->halo > 0 ? taps->halo : 1))
      return fir_pipeline_interleaved(ctx, (const float*)x->data, x->channels, (float*)y->data, L, C, &dprog);
  }
  void *din = nullptr, *dout = nullptr;
  if ((rc = upload(ctx, S_IN, x->data, dx.elems * esize(x->dtype), st, &din)) || (rc = arena(ctx, S_OUT, dy.elems * 4, &dout))) return rc;
  vnd_signal xd = *x, yd = *y;
  xd.data = din;
  yd.data = dout;
  // Wide frame-interleaved float32 slabs: transpose to planar on the device so that the tile loads
  // and stores are coalesced, run the planar kernel, transpose back.
  const bool wide_interleaved = x->dtype == VND_F32 && taps->channels > 2 && x->stride_c == 1 && x->stride_t == x->channels &&
                                x->channels == taps->channels && y->stride_c == 1 && y->stride_t == y->channels && x->frames > 0;
  if (wide_interleaved) {
    void *pin = nullptr, *pout = nullptr;
    if ((rc = arena(ctx, S_WORK, dx.elems * 4, &pin))) return rc;
    if ((rc = arena(ctx, S_AUX, dy.elems * 4, &pout))) return rc;
    if ((rc = transpose_launch((const float*)din, (float*)pin, x->frames, x->channels, st))) return rc;
    vnd_signal xp{pin, x->frames, x->channels, VND_F32, 1, x->frames};
    vnd_signal yp{pout, y->frames, y->channels, VND_F32, 1, y->frames};
    if ((rc = vnd_sparse_fir_dev(&xp, &yp, &dprog, st))) return rc;
    if ((rc = transpose_launch((const float*)pout, (float*)dout, y->channels, y->frames, st))) return rc;
  } else {
    if ((rc = vnd_sparse_fir_dev(&xd, &yd, &dprog, st))) return rc;
  }
  if (dy.elems) VND_CUDA_OK(cudaMemcpyAsync(y->data, dout, dy.elems * 4, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

namespace {

// vnd_vn_decorrelate_host once the context is entered (its lock held, its device current).
int vn_decorrelate_host(vnd_ctx* ctx, const vnd_signal* x, const vnd_signal* out, const vnd_tap_program* taps, const vnd_epilogue* ep) {
  int rc;
  if ((rc = check_vn_decorrelate(x, out, taps, ep))) return rc;
  const Dense dx = dense_extent(x), dy = dense_extent(out);
  VND_REQUIRE(dx.ok && dy.ok, VND_EUNSUPPORTED, "host signals must be contiguous C-order (frames, channels) or planar (channels, frames)");
  cudaStream_t st = ctx->streams[0];
  vnd_tap_program dprog;
  if ((rc = upload_program(ctx, taps, &dprog, st))) return rc;
  void *din = nullptr, *dout = nullptr, *work = nullptr;
  size_t wbytes = 0;
  if ((rc = vnd_vn_decorrelate_workspace(x->frames, taps->channels, ep, &wbytes))) return rc;
  if ((rc = upload(ctx, S_IN, x->data, dx.elems * esize(x->dtype), st, &din)) ||
      (rc = arena(ctx, S_OUT, dy.elems * esize(out->dtype), &dout)) || (rc = arena(ctx, S_WORK, wbytes, &work)))
    return rc;
  vnd_signal xd = *x, od = *out;
  xd.data = din;
  od.data = dout;
  if ((rc = vnd_vn_decorrelate_dev(&xd, &od, &dprog, ep, work, wbytes, st))) return rc;
  if (dy.elems) VND_CUDA_OK(cudaMemcpyAsync(out->data, dout, dy.elems * esize(out->dtype), cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

// 1 + the largest tap index of channel c of a host SEGMENTED program (0 for an empty block or no taps)
int channel_halo(const vnd_tap_program* t, int c) {
  const int32_t* w = t->words + t->offsets[c];
  if (t->offsets[c + 1] == t->offsets[c]) return 0;
  const int S = w[0];
  long long taps = 0;
  for (int s = 0; s < S; ++s) taps += (long long)w[1 + 3 * s] + w[2 + 3 * s];
  int halo = 0;
  for (long long k = 0; k < taps; ++k) halo = w[1 + 3 * S + k] + 1 > halo ? w[1 + 3 * S + k] + 1 : halo;
  return halo;
}

// Clip by clip through vn_decorrelate_host: for filters whose halo does not fit the batched kernel.  Correct, but
// one upload / launch sequence / download per clip.
int batch_host_per_clip(vnd_ctx* ctx, const float* x, const int64_t* offs, int32_t n, const int32_t* prog_of, const vnd_tap_program* taps,
                        const vnd_epilogue* ep, void* out, int32_t out_dtype) {
  const size_t es = esize(out_dtype);
  for (int i = 0; i < n; ++i) {
    const long long L = offs[i + 1] - offs[i];
    const int p = prog_of[i];
    vnd_tap_program sub = *taps;
    sub.offsets = taps->offsets + 2 * p;
    sub.channels = 2;
    const int h0 = channel_halo(taps, 2 * p), h1 = channel_halo(taps, 2 * p + 1);
    sub.halo = h0 > h1 ? h0 : h1;
    const int b0 = sub.offsets[1] - sub.offsets[0], b1 = sub.offsets[2] - sub.offsets[1];
    sub.max_channel_words = b0 > b1 ? b0 : b1;
    vnd_signal xs{const_cast<float*>(x) + 2 * offs[i], L, 2, VND_F32, 2, 1};
    vnd_signal os{reinterpret_cast<char*>(out) + (size_t)(offs[i] + (long long)i * ep->haas_delay) * 2 * es, L + ep->haas_delay, 2, out_dtype,
                  2, 1};
    const int rc = vn_decorrelate_host(ctx, &xs, &os, &sub, ep);
    if (rc) return rc;
  }
  return VND_OK;
}

}  // namespace

extern "C" int vnd_vn_decorrelate_host(vnd_ctx* ctx, const vnd_signal* x, const vnd_signal* out, const vnd_tap_program* taps,
                                       const vnd_epilogue* ep) {
  VND_ENTER(ctx);
  return vn_decorrelate_host(ctx, x, out, taps, ep);
}

extern "C" int vnd_vn_decorrelate_batch_host(vnd_ctx* ctx, const void* x, int32_t x_dtype, int64_t rows, const int64_t* frame_offsets,
                                             int32_t n_clips, const int32_t* program_of_clip, const vnd_tap_program* taps,
                                             const vnd_epilogue* ep, void* out, int32_t out_dtype) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_batch(x, x_dtype, rows, frame_offsets, n_clips, program_of_clip, taps, ep, out, out_dtype))) return rc;
  if (n_clips == 0) return VND_OK;
  const int64_t* offs = frame_offsets;
  if ((rc = check_offsets(offs, n_clips, rows))) return rc;
  const int n_prog = taps->channels / 2;
  for (int i = 0; i < n_clips; ++i)
    VND_REQUIRE(program_of_clip[i] >= 0 && program_of_clip[i] < n_prog, VND_EINVAL, "program_of_clip[%d] = %d is outside [0, %d)", i,
                program_of_clip[i], n_prog);
  const float* xf = reinterpret_cast<const float*>(x);
  if (!batch_fits(taps, rows)) return batch_host_per_clip(ctx, xf, offs, n_clips, program_of_clip, taps, ep, out, out_dtype);

  cudaStream_t st = ctx->streams[0];
  vnd_tap_program dprog;
  if ((rc = upload_program(ctx, taps, &dprog, st))) return rc;
  const int delay = ep->haas_delay;
  const size_t es = esize(out_dtype);
  // chunks of whole clips (clip_chunks, or the whole batch as one), each with its own offsets rebased to its first row
  const bool pipe = pipelined((size_t)rows * 8);
  const std::vector<int> first = pipe ? clip_chunks(offs, n_clips, rows) : std::vector<int>{0, n_clips};
  const int nchunks = (int)first.size() - 1;
  std::vector<long long> meta;  // rebased offsets of every chunk (n_k + 1 each)
  meta.reserve((size_t)n_clips + nchunks);
  long long max_rows = 0, max_out_rows = 0;
  int max_clips = 0;
  for (int k = 0; k < nchunks; ++k) {
    const int a = first[k], b = first[k + 1];
    for (int i = a; i <= b; ++i) meta.push_back(offs[i] - offs[a]);
    const long long r = offs[b] - offs[a];
    max_rows = r > max_rows ? r : max_rows;
    max_out_rows = r + (long long)(b - a) * delay > max_out_rows ? r + (long long)(b - a) * delay : max_out_rows;
    max_clips = b - a > max_clips ? b - a : max_clips;
  }
  const size_t off_bytes = meta.size() * 8;
  void* dmeta = nullptr;
  if ((rc = arena(ctx, S_AUX, off_bytes + (size_t)n_clips * 4, &dmeta))) return rc;
  VND_CUDA_OK(cudaMemcpyAsync(dmeta, meta.data(), off_bytes, cudaMemcpyHostToDevice, st));
  VND_CUDA_OK(cudaMemcpyAsync((char*)dmeta + off_bytes, program_of_clip, (size_t)n_clips * 4, cudaMemcpyHostToDevice, st));
  const int64_t* doffs = reinterpret_cast<const int64_t*>(dmeta);
  const int32_t* dprog_of = reinterpret_cast<const int32_t*>((char*)dmeta + off_bytes);
  const size_t wbytes = vn_batch_workspace_bytes(max_rows, max_clips, ep->rms_normalize);
  auto chunk_of = [&](int k) {
    const int a = first[k], b = first[k + 1];
    const long long r = offs[b] - offs[a];
    return PipeChunk{reinterpret_cast<const char*>(xf + 2 * offs[a]), (size_t)r * 8,
                     reinterpret_cast<char*>(out) + (size_t)(offs[a] + (long long)a * delay) * 2 * es, (size_t)(r + (long long)(b - a) * delay) * 2 * es};
  };
  auto compute = [&](int k, void* din, void* dout, void* work, void*, cudaStream_t cs) {
    const int a = first[k], b = first[k + 1];
    return vnd_vn_decorrelate_batch_dev(din, VND_F32, offs[b] - offs[a], doffs + a + k, b - a, dprog_of + a, &dprog, ep, dout, out_dtype, work,
                                        wbytes, cs);
  };
  if (pipe) {
    VND_CUDA_OK(cudaStreamSynchronize(st));  // the program and the offsets are on the device before the other streams read them
    return run_pipeline(ctx, nchunks, (size_t)max_rows * 8, (size_t)max_out_rows * 2 * es, wbytes, chunk_of, compute);
  }
  const PipeChunk c = chunk_of(0);
  void *din = nullptr, *dout = nullptr, *work = nullptr;
  if ((rc = upload(ctx, S_IN, c.src, c.src_bytes, st, &din)) || (rc = arena(ctx, S_OUT, c.dst_bytes, &dout)) ||
      (rc = arena(ctx, S_WORK, wbytes, &work)) || (rc = compute(0, din, dout, work, nullptr, st)))
    return rc;
  if (c.dst_bytes) VND_CUDA_OK(cudaMemcpyAsync(c.dst, dout, c.dst_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_haas_host(vnd_ctx* ctx, const vnd_signal* x, const vnd_signal* out, int32_t delay, int32_t delayed_channel,
                             int32_t mode_ms, int32_t mono, int32_t use_width, double width) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_haas(x, out, delay, delayed_channel))) return rc;
  const Dense dx = dense_extent(x), dy = dense_extent(out);
  VND_REQUIRE(dx.ok && dy.ok, VND_EUNSUPPORTED, "host signals must be contiguous");
  cudaStream_t st = ctx->streams[0];
  void *din = nullptr, *dout = nullptr;
  if ((rc = upload(ctx, S_IN, x->data, dx.elems * esize(x->dtype), st, &din)) || (rc = arena(ctx, S_OUT, dy.elems * esize(out->dtype), &dout)))
    return rc;
  vnd_signal xd = *x, od = *out;
  xd.data = din;
  od.data = dout;
  if ((rc = vnd_haas_dev(&xd, &od, delay, delayed_channel, mode_ms, mono, use_width, width, st))) return rc;
  if (dy.elems) VND_CUDA_OK(cudaMemcpyAsync(out->data, dout, dy.elems * esize(out->dtype), cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_haas_batch_host(vnd_ctx* ctx, const float* x, int64_t rows, const int64_t* frame_offsets, int32_t n_clips,
                                   const vnd_haas_clip* clips, double* out) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_haas_batch(x, rows, frame_offsets, n_clips, clips))) return rc;
  if (n_clips == 0) return VND_OK;
  const int64_t* offs = frame_offsets;
  if ((rc = check_offsets(offs, n_clips, rows))) return rc;
  // out offsets of every clip and one more (the total)
  std::vector<long long> oo((size_t)n_clips + 1, 0);
  for (int i = 0; i < n_clips; ++i) {
    VND_REQUIRE(clips[i].delay >= 0, VND_EINVAL, "clip %d has a negative delay (%d)", i, clips[i].delay);
    VND_REQUIRE(clips[i].delayed_channel == 0 || clips[i].delayed_channel == 1, VND_EINVAL, "clip %d: delayed_channel must be 0 or 1, is %d", i,
                clips[i].delayed_channel);
    oo[i + 1] = oo[i] + (offs[i + 1] - offs[i]) + clips[i].delay;
  }
  VND_REQUIRE(out != nullptr || oo[n_clips] == 0, VND_EINVAL, "out is null");

  cudaStream_t st = ctx->streams[0];
  const size_t clip_bytes = (size_t)n_clips * sizeof(vnd_haas_clip);
  // chunks of whole clips (clip_chunks, or the whole batch as one), each with its own offsets rebased to its first row:
  // chunk k's frame offsets (n_k + 1) and then its out offsets (n_k) start at meta[2 first[k] + k]
  const bool pipe = pipelined((size_t)rows * 8);
  const std::vector<int> first = pipe ? clip_chunks(offs, n_clips, rows) : std::vector<int>{0, n_clips};
  const int nchunks = (int)first.size() - 1;
  std::vector<long long> meta;
  meta.reserve(2 * (size_t)n_clips + nchunks);
  long long max_rows = 0, max_out_rows = 0;
  for (int k = 0; k < nchunks; ++k) {
    const int a = first[k], b = first[k + 1];
    for (int i = a; i <= b; ++i) meta.push_back(offs[i] - offs[a]);
    for (int i = a; i < b; ++i) meta.push_back(oo[i] - oo[a]);
    max_rows = offs[b] - offs[a] > max_rows ? offs[b] - offs[a] : max_rows;
    max_out_rows = oo[b] - oo[a] > max_out_rows ? oo[b] - oo[a] : max_out_rows;
  }
  void* dmeta = nullptr;
  if ((rc = arena(ctx, S_AUX, clip_bytes + meta.size() * 8, &dmeta))) return rc;
  VND_CUDA_OK(cudaMemcpyAsync(dmeta, clips, clip_bytes, cudaMemcpyHostToDevice, st));
  VND_CUDA_OK(cudaMemcpyAsync((char*)dmeta + clip_bytes, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, st));
  const vnd_haas_clip* dclips = reinterpret_cast<const vnd_haas_clip*>(dmeta);
  const int64_t* dtab = reinterpret_cast<const int64_t*>((char*)dmeta + clip_bytes);
  auto chunk_of = [&](int k) {
    const int a = first[k], b = first[k + 1];
    return PipeChunk{reinterpret_cast<const char*>(x + 2 * offs[a]), (size_t)(offs[b] - offs[a]) * 8, reinterpret_cast<char*>(out + 2 * oo[a]),
                     (size_t)(oo[b] - oo[a]) * 16};
  };
  auto compute = [&](int k, void* din, void* dout, void*, void*, cudaStream_t cs) {
    const int a = first[k], b = first[k + 1];
    const int64_t* tab = dtab + 2 * a + k;
    return vnd_haas_batch_dev(reinterpret_cast<const float*>(din), offs[b] - offs[a], tab, b - a, dclips + a, tab + (b - a + 1), oo[b] - oo[a],
                              reinterpret_cast<double*>(dout), cs);
  };
  if (pipe) {
    VND_CUDA_OK(cudaStreamSynchronize(st));  // the tables are on the device before the other streams read them
    return run_pipeline(ctx, nchunks, (size_t)max_rows * 8, (size_t)max_out_rows * 16, 0, chunk_of, compute);
  }
  const PipeChunk c = chunk_of(0);
  void *din = nullptr, *dout = nullptr;
  if ((rc = upload(ctx, S_IN, c.src, c.src_bytes, st, &din)) || (rc = arena(ctx, S_OUT, c.dst_bytes, &dout)) ||
      (rc = compute(0, din, dout, nullptr, nullptr, st)))
    return rc;
  if (c.dst_bytes) VND_CUDA_OK(cudaMemcpyAsync(c.dst, dout, c.dst_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_stereo_op_host(vnd_ctx* ctx, const vnd_signal* a, const vnd_signal* dry, int32_t op, double width) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_stereo_op(a, dry, op))) return rc;
  const bool with_dry = op == 3 || op == 4;
  const Dense da = dense_extent(a), dd = with_dry ? dense_extent(dry) : Dense{0, true};
  VND_REQUIRE(da.ok && dd.ok, VND_EUNSUPPORTED, "host signals must be contiguous");
  cudaStream_t st = ctx->streams[0];
  void *dA = nullptr, *dD = nullptr, *work = nullptr;
  const size_t wbytes = 64 + colsumsq_workspace_bytes(a->frames);
  if ((rc = upload(ctx, S_IN, a->data, da.elems * esize(a->dtype), st, &dA)) || (rc = arena(ctx, S_WORK, wbytes, &work)) ||
      (with_dry && (rc = upload(ctx, S_OUT, dry->data, dd.elems * esize(dry->dtype), st, &dD))))
    return rc;
  vnd_signal ad = *a, drd = with_dry ? *dry : vnd_signal{};
  ad.data = dA;
  drd.data = dD;
  if ((rc = vnd_stereo_op_dev(&ad, with_dry ? &drd : nullptr, op, width, work, wbytes, st))) return rc;
  if (da.elems) VND_CUDA_OK(cudaMemcpyAsync(a->data, dA, da.elems * esize(a->dtype), cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_vn_objective_batch_host(vnd_ctx* ctx, const float* clips, int64_t frames, int32_t n_clips, int64_t clip_stride,
                                           int64_t chan_stride, const vnd_tap_program* cand, double* partials) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_vn_objective_batch(clips, frames, n_clips, cand, partials))) return rc;
  if (n_clips == 0 || cand->channels == 0) return VND_OK;
  VND_REQUIRE(chan_stride >= frames && clip_stride >= chan_stride + frames, VND_EUNSUPPORTED, "clips must be planar: clip, channel, frame");
  cudaStream_t st = ctx->streams[0];
  vnd_tap_program dprog;
  if ((rc = upload_program(ctx, cand, &dprog, st))) return rc;
  const size_t in_bytes = ((size_t)(n_clips - 1) * clip_stride + chan_stride + frames) * 4;
  const size_t out_bytes = (size_t)n_clips * cand->channels * 12 * 8;
  size_t wbytes = 0;
  if ((rc = vnd_objective_workspace(frames, n_clips, cand->channels, &wbytes))) return rc;
  void *din = nullptr, *dout = nullptr, *work = nullptr;
  if ((rc = upload(ctx, S_IN, clips, in_bytes, st, &din)) || (rc = arena(ctx, S_OUT, out_bytes, &dout)) || (rc = arena(ctx, S_WORK, wbytes, &work)))
    return rc;
  if ((rc = vnd_vn_objective_batch_dev((const float*)din, frames, n_clips, clip_stride, chan_stride, &dprog, (double*)dout, work, wbytes, st)))
    return rc;
  VND_CUDA_OK(cudaMemcpyAsync(partials, dout, out_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_haas_objective_batch_host(vnd_ctx* ctx, const void* clips, int32_t clip_dtype, int64_t frames, int32_t n_clips, int64_t clip_stride,
                                             int64_t chan_stride, const int32_t* delays, int32_t n_cand, double* partials) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_haas_objective_batch(clips, clip_dtype, frames, n_clips, delays, n_cand, partials))) return rc;
  if (n_clips == 0 || n_cand == 0) return VND_OK;
  VND_REQUIRE(chan_stride >= frames && clip_stride >= chan_stride + frames, VND_EUNSUPPORTED, "clips must be planar: clip, channel, frame");
  cudaStream_t st = ctx->streams[0];
  const size_t in_bytes = ((size_t)(n_clips - 1) * clip_stride + chan_stride + frames) * esize(clip_dtype);
  const size_t out_bytes = (size_t)n_clips * n_cand * 8 * 8;
  void *din = nullptr, *dout = nullptr, *dd = nullptr;
  if ((rc = upload(ctx, S_IN, clips, in_bytes, st, &din)) || (rc = arena(ctx, S_OUT, out_bytes, &dout)) ||
      (rc = upload(ctx, S_AUX, delays, (size_t)n_cand * 4, st, &dd)))
    return rc;
  if ((rc = vnd_haas_objective_batch_dev(din, clip_dtype, frames, n_clips, clip_stride, chan_stride, (const int32_t*)dd, n_cand, (double*)dout,
                                         nullptr, 0, st)))
    return rc;
  VND_CUDA_OK(cudaMemcpyAsync(partials, dout, out_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_haas_objective_pairs_host(vnd_ctx* ctx, const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets,
                                             int32_t n_clips, const int32_t* pair_clip, const int32_t* pair_delay, int32_t n_pairs,
                                             double* partials) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_haas_pairs(x, rows, chan_stride, frame_offsets, n_clips, pair_clip, pair_delay, n_pairs, partials))) return rc;
  if (n_pairs == 0) return VND_OK;
  const int64_t* offs = frame_offsets;
  if ((rc = check_offsets(offs, n_clips, rows))) return rc;
  for (int p = 0; p < n_pairs; ++p) {
    const int c = pair_clip[p], d = pair_delay[p];
    VND_REQUIRE(c >= 0 && c < n_clips, VND_EINVAL, "pair_clip[%d] = %d is outside [0, %d)", p, c, n_clips);
    VND_REQUIRE(d >= 0, VND_EINVAL, "pair_delay[%d] = %d is negative", p, d);
    // the reference takes max(|theta|) of the frames: an empty output is a ValueError there (optimization.py:41-43)
    VND_REQUIRE(d > 0 || offs[c + 1] > offs[c], VND_EINVAL,
                "pair %d: objective of an empty signal (clip %d has no frames and delay 0: zero-size array to reduction operation maximum "
                "which has no identity)", p, c);
  }
  cudaStream_t st = ctx->streams[0];
  const size_t in_bytes = rows > 0 ? ((size_t)chan_stride + rows) * 4 : 0;
  const size_t out_bytes = (size_t)n_pairs * 8 * 8;
  const size_t off_bytes = ((size_t)n_clips + 1) * 8, idx_bytes = (size_t)n_pairs * 4;
  void *din = nullptr, *dout = nullptr, *dmeta = nullptr;
  if ((rc = upload(ctx, S_IN, x, in_bytes, st, &din)) || (rc = arena(ctx, S_OUT, out_bytes, &dout)) ||
      (rc = arena(ctx, S_AUX, off_bytes + 2 * idx_bytes, &dmeta)))
    return rc;
  char* meta = reinterpret_cast<char*>(dmeta);
  VND_CUDA_OK(cudaMemcpyAsync(meta, offs, off_bytes, cudaMemcpyHostToDevice, st));
  VND_CUDA_OK(cudaMemcpyAsync(meta + off_bytes, pair_clip, idx_bytes, cudaMemcpyHostToDevice, st));
  VND_CUDA_OK(cudaMemcpyAsync(meta + off_bytes + idx_bytes, pair_delay, idx_bytes, cudaMemcpyHostToDevice, st));
  if ((rc = vnd_haas_objective_pairs_dev((const float*)din, rows, chan_stride, reinterpret_cast<const int64_t*>(meta), n_clips,
                                         reinterpret_cast<const int32_t*>(meta + off_bytes), reinterpret_cast<const int32_t*>(meta + off_bytes + idx_bytes),
                                         n_pairs, (double*)dout, st)))
    return rc;
  VND_CUDA_OK(cudaMemcpyAsync(partials, dout, out_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_vn_stereo_objective_host(vnd_ctx* ctx, const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps,
                                            const vnd_vn_stereo_cand* cands, int32_t n_cand, double* partials) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_vn_stereo(x, frames, chan_stride, taps, cands, n_cand, partials))) return rc;
  if (n_cand == 0) return VND_OK;
  cudaStream_t st = ctx->streams[0];
  size_t wbytes = 0;
  if ((rc = vnd_vn_stereo_objective_workspace(frames, n_cand, &wbytes))) return rc;
  const size_t in_bytes = ((size_t)chan_stride + frames) * 4;
  const size_t out_bytes = (size_t)n_cand * 12 * 8, cand_bytes = (size_t)n_cand * sizeof(vnd_vn_stereo_cand);
  vnd_tap_program dprog;
  void *din = nullptr, *dout = nullptr, *work = nullptr, *dc = nullptr;
  if ((rc = upload_program(ctx, taps, &dprog, st))) return rc;
  if ((rc = upload(ctx, S_IN, x, in_bytes, st, &din)) || (rc = arena(ctx, S_OUT, out_bytes, &dout)) || (rc = arena(ctx, S_WORK, wbytes, &work)) ||
      (rc = upload(ctx, S_AUX, cands, cand_bytes, st, &dc)))
    return rc;
  if ((rc = vnd_vn_stereo_objective_dev((const float*)din, frames, chan_stride, &dprog, (const vnd_vn_stereo_cand*)dc, n_cand, (double*)dout, work,
                                        wbytes, st)))
    return rc;
  VND_CUDA_OK(cudaMemcpyAsync(partials, dout, out_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_vn_stereo_rms_objective_host(vnd_ctx* ctx, const float* x, int64_t frames, int64_t chan_stride, const vnd_tap_program* taps,
                                                const vnd_vn_stereo_cand* cands, int32_t n_cand, float* gains, double* partials) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_vn_stereo_rms(x, frames, chan_stride, taps, cands, n_cand, gains, partials))) return rc;
  if (n_cand == 0) return VND_OK;
  cudaStream_t st = ctx->streams[0];
  size_t wbytes = 0;
  if ((rc = vnd_vn_stereo_rms_objective_workspace(frames, n_cand, &wbytes))) return rc;
  const size_t in_bytes = ((size_t)chan_stride + frames) * 4;
  const size_t out_bytes = (size_t)n_cand * 12 * 8, gain_bytes = (size_t)n_cand * 2 * 4, cand_bytes = (size_t)n_cand * sizeof(vnd_vn_stereo_cand);
  vnd_tap_program dprog;
  void *din = nullptr, *dout = nullptr, *work = nullptr, *dc = nullptr;
  if ((rc = upload_program(ctx, taps, &dprog, st))) return rc;
  if ((rc = upload(ctx, S_IN, x, in_bytes, st, &din)) || (rc = arena(ctx, S_OUT, out_bytes + gain_bytes, &dout)) ||
      (rc = arena(ctx, S_WORK, wbytes, &work)) || (rc = upload(ctx, S_AUX, cands, cand_bytes, st, &dc)))
    return rc;
  float* dgains = reinterpret_cast<float*>(reinterpret_cast<char*>(dout) + out_bytes);  // behind the partials
  if ((rc = vnd_vn_stereo_rms_objective_dev((const float*)din, frames, chan_stride, &dprog, (const vnd_vn_stereo_cand*)dc, n_cand, dgains,
                                            (double*)dout, work, wbytes, st)))
    return rc;
  VND_CUDA_OK(cudaMemcpyAsync(partials, dout, out_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaMemcpyAsync(gains, dgains, gain_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_haas_effect_objective_host(vnd_ctx* ctx, const float* x, int64_t frames, int64_t chan_stride, const vnd_haas_clip* cands,
                                              int32_t n_cand, double* partials) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_family_clip(x, frames, chan_stride, cands, n_cand, partials))) return rc;
  for (int i = 0; i < n_cand; ++i) {
    VND_REQUIRE(cands[i].delay >= 0, VND_EINVAL, "candidate %d: negative delay %d", i, cands[i].delay);
    VND_REQUIRE(cands[i].delayed_channel == 0 || cands[i].delayed_channel == 1, VND_EINVAL, "candidate %d: delayed_channel %d is not 0 or 1", i,
                cands[i].delayed_channel);
  }
  if (n_cand == 0) return VND_OK;
  cudaStream_t st = ctx->streams[0];
  const size_t in_bytes = ((size_t)chan_stride + frames) * 4;
  const size_t out_bytes = (size_t)n_cand * 8 * 8, cand_bytes = (size_t)n_cand * sizeof(vnd_haas_clip);
  void *din = nullptr, *dout = nullptr, *dc = nullptr;
  if ((rc = upload(ctx, S_IN, x, in_bytes, st, &din)) || (rc = arena(ctx, S_OUT, out_bytes, &dout)) ||
      (rc = upload(ctx, S_AUX, cands, cand_bytes, st, &dc)))
    return rc;
  if ((rc = vnd_haas_effect_objective_dev((const float*)din, frames, chan_stride, (const vnd_haas_clip*)dc, n_cand, (double*)dout, st))) return rc;
  VND_CUDA_OK(cudaMemcpyAsync(partials, dout, out_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

extern "C" int vnd_vn_objective_runs_host(vnd_ctx* ctx, const float* x, int64_t rows, int64_t chan_stride, const int64_t* frame_offsets,
                                          int32_t n_clips, const vnd_tap_program* cand, const int32_t* run_clip, const int32_t* run_cand,
                                          const int32_t* run_count, const int32_t* run_out, int32_t n_runs, double* partials,
                                          int64_t n_partial_rows) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_runs(x, rows, chan_stride, frame_offsets, n_clips, cand, run_clip, run_cand, run_count, run_out, n_runs, partials,
                       n_partial_rows)))
    return rc;
  if (n_partial_rows == 0) return VND_OK;
  cudaStream_t st = ctx->streams[0];
  size_t wbytes = 0;
  if ((rc = vnd_vn_objective_runs_workspace(frame_offsets, n_clips, run_clip, run_count, n_runs, &wbytes))) return rc;
  const size_t in_bytes = rows > 0 ? ((size_t)chan_stride + rows) * 4 : 0;
  const size_t out_bytes = (size_t)n_partial_rows * 12 * 8;
  vnd_tap_program dprog;
  void *din = nullptr, *dout = nullptr, *work = nullptr;
  if ((rc = upload_program(ctx, cand, &dprog, st))) return rc;
  if ((rc = upload(ctx, S_IN, x, in_bytes, st, &din)) || (rc = arena(ctx, S_OUT, out_bytes, &dout)) || (rc = arena(ctx, S_WORK, wbytes, &work)))
    return rc;
  VND_CUDA_OK(cudaMemsetAsync(dout, 0, out_bytes, st));  // rows no run names come back as zeros
  if ((rc = vnd_vn_objective_runs_dev((const float*)din, rows, chan_stride, frame_offsets, n_clips, &dprog, run_clip, run_cand, run_count, run_out,
                                      n_runs, (double*)dout, n_partial_rows, work, wbytes, st)))
    return rc;
  VND_CUDA_OK(cudaMemcpyAsync(partials, dout, out_bytes, cudaMemcpyDeviceToHost, st));
  VND_CUDA_OK(cudaStreamSynchronize(st));
  return VND_OK;
}

// Streaming planar FIR with an explicit stage size: channel groups flow through the 3-deep ring of run_pipeline
// (upload, kernels and download on three streams; pageable buffers staged through page-locked memory by helper
// threads).  vnd_sparse_fir_host takes the same path for any large float32 slab, planar or (frames, channels).
extern "C" int vnd_sparse_fir_stream_host(vnd_ctx* ctx, const float* x, float* y, int64_t frames, int32_t channels,
                                          const vnd_tap_program* taps, int32_t channels_per_chunk) {
  VND_ENTER(ctx);
  int rc;
  if ((rc = check_taps(taps))) return rc;
  VND_REQUIRE(frames >= 0 && channels >= 0, VND_EINVAL, "negative extent");
  VND_REQUIRE(taps->channels == channels, VND_EINVAL, "tap program has %d channels, slab has %d", taps->channels, channels);
  if (frames == 0 || channels == 0) return VND_OK;
  VND_REQUIRE(x != nullptr && y != nullptr, VND_EINVAL, "null slab");
  vnd_tap_program dprog;
  if ((rc = upload_program(ctx, taps, &dprog, ctx->streams[0]))) return rc;
  VND_CUDA_OK(cudaStreamSynchronize(ctx->streams[0]));
  return fir_pipeline_planar(ctx, x, y, frames, channels, &dprog, channels_per_chunk <= 0 ? 1 : channels_per_chunk);
}
