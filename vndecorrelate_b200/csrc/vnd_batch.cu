// Batched VelvetNoise.decorrelate (+ LR Haas) over many clips of different lengths packed in one (rows, 2) float32
// array (vnd_vn_decorrelate_batch_dev).  A fixed number of launches per batch, whatever the number of clips:
//   no normaliser : vn_batch_stereo_kernel (vnd_fir.cu) writes the final output, Haas placement and zero fill included;
//   rms_normalize : vn_batch_stereo_kernel writes a float32 scratch, then the order-exact sums of squares of the 4 columns
//                   of every clip (batch_sumsq_serial_kernel, or the cluster scan of vnd_post.cu for few long columns),
//                   ending with each clip's gains computed as rms_gain_kernel does, then batch_place_kernel places the scaled result.
// Every clip's bytes are those of the single-clip path (vnd_vn_decorrelate_dev) on that clip.

#include <math.h>

#include "vnd_batch.cuh"

namespace vnd {

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------------------------------------
// Many columns: the four running sums of a clip (x0, x1, y0, y1) are four independent dependent-add chains of one
// thread, so they cost what one chain costs (~4 clocks per row).  One CTA per clip: warps 1..7 stage the rounded
// squares of the next chunk of rows (one float4 per row; the loads of the interleaved pairs coalesce) while lane 0 of
// warp 0 walks the current chunk.  Rows past the clip's end are +0: s + 0 == s.
// ------------------------------------------------------------------------------------------------
constexpr int kSerChunk = 1024;  // rows per stage: 2 x 16 KB of static shared memory, 7 CTAs per SM

__global__ void __launch_bounds__(256) batch_sumsq_serial_kernel(const BatchSumCols c) {
  constexpr int NT = 256;
  __shared__ __align__(16) float4 buf[2][kSerChunk];
  const int clip = blockIdx.x;
  const int tid = threadIdx.x;
  const long long o = c.offs[clip];
  const long long L = c.offs[clip + 1] - o;
  const float2* __restrict__ x2 = reinterpret_cast<const float2*>(c.x) + o;
  const float2* __restrict__ y2 = reinterpret_cast<const float2*>(c.y) + o;
  const long long nchunks = L > 0 ? ceil_div<long long>(L, kSerChunk) : 0;
  auto stage = [&](long long k, int slot, int first, int step) {
    const long long off = k * kSerChunk;
    for (int i = first; i < kSerChunk; i += step) {
      const long long t = off + i;
      float4 v = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      if (t < L) {
        const float2 a = x2[t], b = y2[t];
        v = make_float4(fmul(a.x, a.x), fmul(a.y, a.y), fmul(b.x, b.x), fmul(b.y, b.y));
      }
      buf[slot][i] = v;
    }
  };
  if (nchunks > 0) stage(0, 0, tid, NT);
  float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
  for (long long k = 0; k < nchunks; ++k) {
    __syncthreads();
    if (tid < 32) {
      if (tid == 0) {
        const float4* q = buf[k & 1];
        const long long left = L - k * kSerChunk;
        const int n = (int)(left < kSerChunk ? left : kSerChunk);
        const int n8 = (n + 7) & ~7;
#pragma unroll 2
        for (int i = 0; i < n8; i += 8) {
          float4 v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = q[i + j];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            s0 = fadd(s0, v[j].x);
            s1 = fadd(s1, v[j].y);
            s2 = fadd(s2, v[j].z);
            s3 = fadd(s3, v[j].w);
          }
        }
      }
    } else if (k + 1 < nchunks) {
      stage(k + 1, (int)((k + 1) & 1), tid - 32, NT - 32);
    }
  }
  if (tid == 0) c.store_clip(clip, s0, s1, s2, s3);
}

// ------------------------------------------------------------------------------------------------
// Placement: each CTA takes one (clip, tile) pair (batch_clip_of) and writes the rows scaled by its clip's two gains
// (computed by the sums pass with the clip's own frame count, as rms_gain_kernel does), delayed, and the clip's Haas
// zero fill.
// ------------------------------------------------------------------------------------------------
struct BatchPlaceParams {
  const float* y;  // packed (rows, 2) scratch
  const long long* offs;
  const float* gains;  // 2 per clip
  void* out;          // (rows + n delay, 2)
  int n_clips;
  int delay, delay_ch;
};

template <typename TOut>
__global__ void __launch_bounds__(256) batch_place_kernel(const BatchPlaceParams p) {
  constexpr int NT = 256;
  const int clip = batch_clip_of(p.offs, p.n_clips, kBatchTile, blockIdx.x);
  const long long c0 = p.offs[clip];
  const long long L = p.offs[clip + 1] - c0;
  const long long k = (long long)blockIdx.x - (c0 / kBatchTile + clip);
  const long long ntiles = L > 0 ? ceil_div<long long>(L, kBatchTile) : 1;
  if (k < 0 || k >= ntiles) return;
  const float g0 = p.gains[2 * (long long)clip], g1 = p.gains[2 * (long long)clip + 1];
  TOut* __restrict__ out = reinterpret_cast<TOut*>(p.out) + 2 * (c0 + (long long)clip * p.delay);
  const float2* __restrict__ y2 = reinterpret_cast<const float2*>(p.y) + c0;
  const int sh0 = p.delay_ch == 0 ? p.delay : 0;
  const int sh1 = p.delay_ch == 1 ? p.delay : 0;
  const long long t0 = k * kBatchTile;
  for (int i = threadIdx.x; i < kBatchTile; i += NT) {
    const long long t = t0 + i;
    if (t < L) {
      const float2 v = y2[t];
      out[(t + sh0) * 2] = (TOut)fmul(v.x, g0);
      out[(t + sh1) * 2 + 1] = (TOut)fmul(v.y, g1);
    }
  }
  if (p.delay > 0) {
    if (k == 0)
      for (int i = threadIdx.x; i < p.delay; i += NT) out[(long long)i * 2 + p.delay_ch] = (TOut)0;
    if (k == ntiles - 1)
      for (int i = threadIdx.x; i < p.delay; i += NT) out[(L + i) * 2 + (1 - p.delay_ch)] = (TOut)0;
  }
}

// ------------------------------------------------------------------------------------------------
// Batched HaasEffect.decorrelate (vnd_haas_batch_dev): each CTA takes one (clip, output tile) pair (batch_clip_of over
// the out offsets) and writes every output frame of its tile, the clip's head and tail zeros included, as one double2;
// the two input frames it reads (undelayed and delayed) are float2 loads that coalesce across the warp.  The second
// read of each input frame comes `delay` frames later, from L1 or L2.
// ------------------------------------------------------------------------------------------------
static_assert(sizeof(vnd_haas_clip) == 32, "vnd_haas_clip is two 16-byte words");

struct HaasBatchParams {
  const float* x;               // packed (rows, 2)
  const long long* offs;        // n + 1
  const long long* out_offs;    // n
  const vnd_haas_clip* clips;   // n, 16-byte aligned
  double* out;                  // (out_rows, 2)
  int n_clips;
};

__global__ void __launch_bounds__(256) haas_batch_kernel(const HaasBatchParams p) {
  constexpr int NT = 256;
  const int clip = batch_clip_of(p.out_offs, p.n_clips, kHaasTile, blockIdx.x);
  const long long o0 = p.out_offs[clip];
  const long long k = (long long)blockIdx.x - (o0 / kHaasTile + clip);
  const int4* rec = reinterpret_cast<const int4*>(p.clips + clip);
  const int4 w0 = __ldg(rec), w1 = __ldg(rec + 1);
  const int delay = w0.x, dch = w0.y, mode_ms = w0.z, mono = w0.w, use_width = w1.x;
  const double width = __hiloint2double(w1.w, w1.z);
  const long long x0 = p.offs[clip];
  const long long L = p.offs[clip + 1] - x0;
  const long long t0 = k * kHaasTile;
  const long long t1 = t0 + kHaasTile < L + delay ? t0 + kHaasTile : L + delay;
  if (k < 0 || t0 >= t1) return;
  const float2* __restrict__ x2 = reinterpret_cast<const float2*>(p.x) + x0;
  double2* __restrict__ o2 = reinterpret_cast<double2*>(p.out) + o0;
  const int sh0 = dch == 0 ? delay : 0, sh1 = dch == 1 ? delay : 0;
#pragma unroll 4
  for (long long m = t0 + threadIdx.x; m < t1; m += NT) {
    const long long q0 = m - sh0, q1 = m - sh1;
    const bool v0 = q0 >= 0 && q0 < L, v1 = q1 >= 0 && q1 < L;
    float2 s0 = make_float2(0.0f, 0.0f), s1 = make_float2(0.0f, 0.0f);
    if (v0) s0 = __ldg(x2 + q0);
    if (v1) s1 = __ldg(x2 + q1);
    o2[m] = haas_frame(s0.x, s0.y, v0, s1.x, s1.y, v1, mode_ms, mono, use_width, width);
  }
}

int haas_batch_launch(const float* x, const long long* offs, int n_clips, const vnd_haas_clip* clips, const long long* out_offs,
                      long long out_rows, double* out, cudaStream_t st) {
  if (n_clips == 0 || out_rows == 0) return VND_OK;
  const long long blocks = out_rows / kHaasTile + n_clips;
  VND_REQUIRE(blocks < 0x7fffffffLL, VND_EUNSUPPORTED, "grid too large (%lld CTAs)", blocks);
  const HaasBatchParams p{x, offs, out_offs, clips, out, n_clips};
  haas_batch_kernel<<<(unsigned)blocks, 256, 0, st>>>(p);
  return after_launch("haas_batch_kernel");
}

// ------------------------------------------------------------------------------------------------
// One Haas step of many live signals (vnd_haas_block_step_dev): signal i's output frames [T0, T0 + count) are those of
// HaasEffect.decorrelate on its whole input, because output frame m reads input frames m - sh0, m - sh1 <= m only.
// A frame at or past T1 is +0 and not valid, as past the end of a one-shot signal of T1 frames: a final step's tail.
// ------------------------------------------------------------------------------------------------
bool block_step_grid(BlockStepParams* b, long long out_rows, int tile, long long* blocks) {
  b->out_blocks = out_rows / tile + b->n;
  b->hchunks = (b->H + kHistTile - 1) / kHistTile;
  *blocks = b->out_blocks + (long long)b->n * b->hchunks;
  return *blocks < 0x7fffffffLL;
}

__global__ void __launch_bounds__(256) haas_block_step_kernel(const BlockStepParams b, const vnd_haas_clip* clips, double* out) {
  constexpr int NT = 256;
  if (blockIdx.x >= b.out_blocks) {
    block_step_history(b, (long long)blockIdx.x - b.out_blocks);
    return;
  }
  const int sig = batch_clip_of(b.out_offs, b.n, kHaasTile, blockIdx.x);
  const long long o0 = b.out_offs[sig];
  const long long cnt = b.out_offs[sig + 1] - o0;
  const long long k = (long long)blockIdx.x - (o0 / kHaasTile + sig);
  const long long j0 = k * kHaasTile;
  if (k < 0 || j0 >= cnt) return;
  const long long j1 = j0 + kHaasTile < cnt ? j0 + kHaasTile : cnt;
  const int4* rec = reinterpret_cast<const int4*>(clips + sig);
  const int4 w0 = __ldg(rec), w1 = __ldg(rec + 1);
  const int delay = w0.x, dch = w0.y, mode_ms = w0.z, mono = w0.w, use_width = w1.x;
  const double width = __hiloint2double(w1.w, w1.z);
  const long long T0 = b.received[sig], x0 = b.offs[sig];
  const long long T1 = T0 + (b.offs[sig + 1] - x0);
  double2* __restrict__ o2 = reinterpret_cast<double2*>(out) + o0;
  const int sh0 = dch == 0 ? delay : 0, sh1 = dch == 1 ? delay : 0;
  for (long long j = j0 + threadIdx.x; j < j1; j += NT) {
    const long long q0 = T0 + j - sh0, q1 = T0 + j - sh1;
    const bool v0 = q0 >= 0 && q0 < T1, v1 = q1 >= 0 && q1 < T1;
    const float2 s0 = block_step_frame(b, sig, q0, T0, T1, x0);
    const float2 s1 = block_step_frame(b, sig, q1, T0, T1, x0);
    o2[j] = haas_frame(s0.x, s0.y, v0, s1.x, s1.y, v1, mode_ms, mono, use_width, width);
  }
}

int haas_block_step_launch(BlockStepParams b, long long out_rows, const vnd_haas_clip* clips, double* out, cudaStream_t st) {
  long long blocks = 0;
  VND_REQUIRE(block_step_grid(&b, out_rows, kHaasTile, &blocks), VND_EUNSUPPORTED, "grid too large (%lld CTAs)", blocks);
  haas_block_step_kernel<<<(unsigned)blocks, 256, 0, st>>>(b, clips, out);
  return after_launch("haas_block_step_kernel");
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
size_t vn_batch_workspace_bytes(long long rows, int n_clips, int rms) {
  if (!rms) return 0;
  // sums of the 4 columns, 2 gains and a column counter per clip | float32 scratch of the FIR / M/S / width result
  return align_up((size_t)n_clips * 7 * sizeof(float), 256) + (size_t)rows * 2 * sizeof(float);
}

// Serial chains or the cluster scan, from the shape alone (the clip lengths stay on the device).  A serial chain costs
// about 4 clocks per row and all clips run at once while they fit on the GPU (7 CTAs per SM); the scan costs PS_K CTAs
// per column and a round of about 6000 clocks per PS_K x 8192 rows.  Both give the same bits.
static bool use_cluster_scan(long long rows, int n_clips, int sm_count) {
  const double per_clip = (double)rows / n_clips;
  const int k = seq_sumsq_cluster_width();
  if (per_clip < (double)seq_sumsq_scan_head() + 2.0 * seq_sumsq_scan_round()) return false;
  const double serial = ceil((double)n_clips / (7.0 * sm_count)) * per_clip * 4.0;
  const double scan = ceil(4.0 * n_clips * k / sm_count) * ceil(per_clip / ((double)k * seq_sumsq_scan_round())) * 6000.0;
  return scan < serial;
}

int vn_batch_launch(const float* x, long long rows, const long long* offs, int n_clips, const int* prog_of, const vnd_tap_program* taps,
                    const vnd_epilogue* ep, void* out, int out_dtype, void* workspace, cudaStream_t st) {
  if (n_clips == 0) return VND_OK;
  const int delay = ep->haas_delay, dch = ep->haas_channel;
  if (!ep->rms_normalize) return vn_batch_stereo_launch(x, rows, offs, n_clips, prog_of, taps, ep, out, out_dtype, delay, dch, nullptr, st);
  char* ws = reinterpret_cast<char*>(workspace);
  float* sums = reinterpret_cast<float*>(ws);
  float* gains = sums + 4 * (size_t)n_clips;
  unsigned* arrivals = reinterpret_cast<unsigned*>(gains + 2 * (size_t)n_clips);
  float* scratch = reinterpret_cast<float*>(ws + align_up((size_t)n_clips * 7 * sizeof(float), 256));
  int rc;
  if ((rc = vn_batch_stereo_launch(x, rows, offs, n_clips, prog_of, taps, ep, scratch, VND_F32, 0, 0, arrivals, st))) return rc;
  const BatchSumCols cols{x, scratch, offs, sums, gains, arrivals};
  DeviceInfo di;
  if ((rc = device_info(&di))) return rc;
  if (use_cluster_scan(rows, n_clips, di.sm_count)) {
    if ((rc = batch_sumsq_cluster_launch(cols, 4 * n_clips, st))) return rc;
  } else {
    batch_sumsq_serial_kernel<<<(unsigned)n_clips, 256, 0, st>>>(cols);
    if ((rc = after_launch("batch_sumsq_serial_kernel"))) return rc;
  }
  BatchPlaceParams p{};
  p.y = scratch;
  p.offs = offs;
  p.gains = gains;
  p.out = out;
  p.n_clips = n_clips;
  p.delay = delay;
  p.delay_ch = dch;
  const long long blocks = rows / kBatchTile + n_clips;
  VND_REQUIRE(blocks < 0x7fffffffLL, VND_EUNSUPPORTED, "grid too large (%lld CTAs)", blocks);
  if (out_dtype == VND_F64) batch_place_kernel<double><<<(unsigned)blocks, 256, 0, st>>>(p);
  else batch_place_kernel<float><<<(unsigned)blocks, 256, 0, st>>>(p);
  return after_launch("batch_place_kernel");
}

}  // namespace vnd
