// awm_capi.cu -- implementation of the C ABI declared in include/awm_b200.h.
//
// One context = one device + one stream + growable device buffers.  Host pointers are staged
// through context-owned device memory; device pointers are used in place.  There is no CPU
// fallback: every entry point launches the sm_100a kernels of awm_kernels.cuh or fails.
#include "awm_kernels.cuh"
#include "awm_speed.cuh"
#include "awm_wav_decode.cuh"
#include "awm_refine_slide.cuh"
#include "awm_approx_mags.cuh"
#include <vector>
#include <time.h>
#include <string.h>
#include "awm_approx_tc.cuh"
#include "awm_embed_strip.cuh"
#include "awm_viterbi_pair.cuh"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <algorithm>
#include <map>
#include <thread>
#include <limits.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

using namespace awm;

namespace {

struct DevBuf
{
  void  *p = nullptr;
  size_t cap = 0;
  cudaError_t
  reserve (size_t bytes)
  {
    if (bytes <= cap)
      return cudaSuccess;
    if (p)
      cudaFree (p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc (&p, want);
    if (e == cudaSuccess)
      cap = want;
    return e;
  }
  void
  release()
  {
    if (p)
      cudaFree (p);
    p = nullptr;
    cap = 0;
  }
  template<class T> T *as() { return static_cast<T *> (p); }
};

/* page-locked staging memory for the small lists that go back and forth between the stages of a `get` (candidate lists, per-offset
 * sums, soft bits, code words): copies from / to pageable memory are staged by the driver and block the host; with pinned memory
 * the copies of a stage are queued back to back and cost one synchronisation.  Bump allocator, reset at the start of an API call. */
struct PinArena
{
  struct Chunk { unsigned char *p; size_t cap; };
  std::vector<Chunk> chunks;
  size_t cur = 0, off = 0;
  void reset() { cur = 0; off = 0; }
  void *alloc (size_t n)
  {
    n = (n + 63) & ~size_t (63);
    for (;;)
      {
        if (cur < chunks.size() && off + n <= chunks[cur].cap)
          {
            void *r = chunks[cur].p + off;
            off += n;
            return r;
          }
        if (cur + 1 < chunks.size())
          {
            cur++;
            off = 0;
            continue;
          }
        Chunk c { nullptr, std::max<size_t> (n, size_t (4) << 20) };
        if (cudaMallocHost (reinterpret_cast<void **> (&c.p), c.cap) != cudaSuccess)
          return nullptr;
        chunks.push_back (c);
        cur = chunks.size() - 1;
        off = 0;
      }
  }
  template<class T> T *get (size_t count) { return static_cast<T *> (alloc (std::max<size_t> (count, 1) * sizeof (T))); }
  void release()
  {
    for (auto& c : chunks)
      cudaFreeHost (c.p);
    chunks.clear();
    reset();
  }
};

inline double
wall_now()
{
  timespec ts;
  clock_gettime (CLOCK_MONOTONIC, &ts);
  return double (ts.tv_sec) + 1e-9 * double (ts.tv_nsec);
}

struct SyncTab
{
  DevBuf ent, off, sorted, groups;
  DevBuf masks, masks48, masks64;     // 0/1 band masks of the entries as tcgen05 B operand chunks of 128 / 48 / 64 entries (awm_approx_tc.cuh)
  int n_chunks = 0, n_chunks48 = 0, n_chunks64 = 0;
  int n_groups = 0;
  int n_ent = 0, n_bits = 0, total_frames = 0;
  std::vector<awm_sync_entry> h_ent;
  std::vector<int> h_off;
};

struct KeyTab
{
  SyncTab sync[2];
  DevBuf mix, order;
  int n_mix = 0, n_coded = 0, frames_per_bit = 0, fpb = 0;
};

/* sample layouts of the PCM entry points: the float pipeline's own samples (no conversion), or stored WAV samples (WavSampleType) */
constexpr int kPcmFloat = -1;

} // namespace

struct awm_ctx
{
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t s_in = nullptr, s_out = nullptr;      // copy streams of the pipelined host paths
  std::string err;
  uint64_t launches = 0;
  int n_sms = 0;
  bool profiling = false;
  struct ProfRec { const char *name; cudaEvent_t e0, e1; double bytes; };
  std::vector<ProfRec> prof;

  DevBuf tw, win, synth;             // constant tables
  DevBuf frame_mod; int embed_fpb = 0;
  KeyTab keys[AWM_MAX_KEYS];

  // bound PCM
  const float *pcm = nullptr; size_t pcm_frames = 0; int pcm_ch = 0;
  DevBuf pcm_own, pcm16_own;
  /* one prefetched span.  type kPcmFloat: buf holds the copy; a WAV sample type: raw holds the stored bytes, they become float in buf
   * when the span is bound, and stay in raw (the next span may take its head from there) until the slot is prefetched into again */
  struct Prefetch { DevBuf buf, raw; int type = kPcmFloat; const void *src = nullptr; size_t n_frames = 0; int ch = 0; cudaEvent_t done = nullptr; bool valid = false, filled = false; };
  Prefetch pref[2];
  int pref_next = 0;
  /* awm_pcm_stage: a host stream on its way into `staged` piece by piece */
  DevBuf staged, staged16;
  std::vector<cudaEvent_t> stage_done;           // one per piece, recorded on s_in
  size_t stage_piece = 0, stage_frames = 0, stage_converted = 0;
  int stage_ch = 0;
  bool stage_s16 = false;

  DevBuf dbT, have, q, scores, a_ud, a_cnt, peaks_out, peaks_cnt, a_mags;       // approx
  size_t n_scores_dev = 0;
  DevBuf cand_start, cand_noff, r_ud, r_cnt, rvalid, r_ent_ud, r_ent_flag, tw1024;   // refine
  DevBuf blk_start, D, raw;          // decode
  DevBuf vit_raw, vit_off, vit_types, vit_delta, vit_dec, vit_bits, vit_err, vit_order;
  DevBuf emb_in, emb_out, emb_in16, emb_out16, peaks, snr;

  PinArena pin;

  // multi-GPU exchange (awm_dist_*): NCCL communicator of the sharded run + staging buffers
  void *nccl_comm = nullptr;
  int dist_rank = 0, dist_world = 1;
  DevBuf dist_send, dist_recv;
  unsigned char *dist_hsend = nullptr, *dist_hhdr = nullptr;
  size_t dist_hsend_cap = 0;

  // resampler / speed scan
  struct CoefTab { DevBuf buf; int h = 0; };
  std::map<std::pair<double, int>, CoefTab> coef_cache;          // (ratio, hlen) -> filter table
  DevBuf rs_in, rs_out, rs_jobs, pcm_rs;
  const float *saved_pcm = nullptr; size_t saved_frames = 0; int saved_ch = 0; bool pushed = false;
  DevBuf win512, sp_clip, sp_sub, sp_mags, sp_mag_jobs, sp_cmp_jobs, sp_best;
};

namespace {

int
fail (awm_ctx *ctx, const char *fmt, ...)
{
  char buf[512];
  va_list ap;
  va_start (ap, fmt);
  vsnprintf (buf, sizeof (buf), fmt, ap);
  va_end (ap);
  if (ctx)
    ctx->err = buf;
  return 1;
}

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail (ctx, "%s: %s", #call, cudaGetErrorString (e_)); } while (0)
#define LAUNCH_CHECK(name) do { ctx->launches++; cudaError_t e_ = cudaGetLastError(); if (e_ != cudaSuccess) return fail (ctx, "launch %s: %s", name, cudaGetErrorString (e_)); prof_end (ctx, name); } while (0)
/* PROF (ctx) goes right before a kernel launch, LAUNCH_CHECK right after it */
#define PROF(ctx) prof_begin (ctx)

void
prof_begin (awm_ctx *ctx)
{
  if (!ctx->profiling)
    return;
  awm_ctx::ProfRec r;
  r.name = nullptr;
  r.bytes = 0;
  cudaEventCreate (&r.e0);
  cudaEventCreate (&r.e1);
  cudaEventRecord (r.e0, ctx->stream);
  ctx->prof.push_back (r);
}

void
prof_end (awm_ctx *ctx, const char *name)
{
  if (!ctx->profiling || ctx->prof.empty() || ctx->prof.back().name)
    return;
  ctx->prof.back().name = name;
  cudaEventRecord (ctx->prof.back().e1, ctx->stream);
}

/* measurement aid: algorithmic bytes of the launch that was just recorded (the compulsory traffic of the work it was given;
 * only kernels whose volume depends on run-time counts report it here, the others are sized by the caller from the input) */
void
prof_bytes (awm_ctx *ctx, double bytes)
{
  if (ctx->profiling && !ctx->prof.empty())
    ctx->prof.back().bytes = bytes;
}

bool
is_device_ptr (const void *p)
{
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes (&a, p) != cudaSuccess)
    {
      cudaGetLastError();
      return false;
    }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

int
pcm_sample_bytes (int type)
{
  switch (type)
    {
    case WAV_U8:  return 1;
    case WAV_S16: return 2;
    case WAV_S24: return 3;
    case WAV_F64: return 8;
    default:      return 4;
    }
}

/* awm_wav_format -> WavSampleType; -1 for a format no WAV input of `get` can have */
int
wav_sample_type (awm_wav_format f)
{
  if (f.is_float)
    return f.bits == 32 ? WAV_F32 : f.bits == 64 ? WAV_F64 : -1;
  switch (f.bits)
    {
    case 8:  return WAV_U8;
    case 16: return WAV_S16;
    case 24: return WAV_S24;
    case 32: return WAV_S32;
    default: return -1;
    }
}

/* k_wav_to_f32 for a sample type known at run time: n samples at `in` (any byte address) -> out.  Profiled when it runs on the
 * context stream (the profile events live there). */
int
wav_to_f32 (awm_ctx *ctx, int type, const void *in, float *out, long long n, cudaStream_t st)
{
  if (n <= 0)
    return 0;
  const unsigned grid = unsigned (((n + 3) / 4 + 255) / 256);
  const unsigned char *b = static_cast<const unsigned char *> (in);
  if (st == ctx->stream)
    PROF (ctx);
  switch (type)
    {
    case WAV_U8:  k_wav_to_f32<WAV_U8><<<grid, 256, 0, st>>> (b, out, n);  LAUNCH_CHECK ("k_wav_to_f32<u8>");  break;
    case WAV_S16: k_wav_to_f32<WAV_S16><<<grid, 256, 0, st>>> (b, out, n); LAUNCH_CHECK ("k_wav_to_f32<s16>"); break;
    case WAV_S24: k_wav_to_f32<WAV_S24><<<grid, 256, 0, st>>> (b, out, n); LAUNCH_CHECK ("k_wav_to_f32<s24>"); break;
    case WAV_S32: k_wav_to_f32<WAV_S32><<<grid, 256, 0, st>>> (b, out, n); LAUNCH_CHECK ("k_wav_to_f32<s32>"); break;
    case WAV_F32: k_wav_to_f32<WAV_F32><<<grid, 256, 0, st>>> (b, out, n); LAUNCH_CHECK ("k_wav_to_f32<f32>"); break;
    case WAV_F64: k_wav_to_f32<WAV_F64><<<grid, 256, 0, st>>> (b, out, n); LAUNCH_CHECK ("k_wav_to_f32<f64>"); break;
    default:      return fail (ctx, "wav_to_f32: unknown sample type %d", type);
    }
  return 0;
}

double
window_cos (double x)    // von Hann, reference src/wmcommon.hh:187-193
{
  if (fabs (x) > 1)
    return 0;
  return 0.5 * cos (x * M_PI) + 0.5;
}

int
init_tables (awm_ctx *ctx)
{
  // twiddles exp(-2 pi i k1 t / 1024) at [k1*32 + t]
  std::vector<float2> tw (1024);
  for (int k1 = 0; k1 < 32; k1++)
    for (int t = 0; t < 32; t++)
      {
        const double a = -2.0 * M_PI * double (k1 * t) / 1024.0;
        tw[k1 * 32 + t] = make_float2 (float (cos (a)), float (sin (a)));
      }
  // FFTAnalyzer::gen_normalized_window (src/wmcommon.cc:68-89)
  std::vector<float> win (kFrame);
  double weight = 0;
  for (int i = 0; i < kFrame; i++)
    {
      const double w = window_cos ((i - kFrame / 2.0) / (kFrame / 2.0));
      win[i] = w;
      weight += w;
    }
  for (int i = 0; i < kFrame; i++)
    win[i] *= 2.0 / weight;
  // WatermarkSynth::generate_window (src/wmadd.cc:177-206)
  std::vector<float> synth (3 * kFrame);
  for (int i = 0; i < 3 * kFrame; i++)
    {
      const double overlap = 0.1;
      double norm_pos = (double (i) - kFrame) / kFrame;
      if (norm_pos > 0.5)
        norm_pos = 1 - norm_pos;
      double tri;
      if (norm_pos < -overlap)
        tri = 0;
      else if (norm_pos < overlap)
        tri = 0.5 + norm_pos / (2 * overlap);
      else
        tri = 1;
      synth[i] = (cos (tri * M_PI + M_PI) + 1) * 0.5;
    }
  CK (ctx->tw.reserve (tw.size() * sizeof (float2)));
  CK (ctx->win.reserve (win.size() * sizeof (float)));
  CK (ctx->synth.reserve (synth.size() * sizeof (float)));
  CK (cudaMemcpy (ctx->tw.p, tw.data(), tw.size() * sizeof (float2), cudaMemcpyHostToDevice));
  CK (cudaMemcpy (ctx->win.p, win.data(), win.size() * sizeof (float), cudaMemcpyHostToDevice));
  CK (cudaMemcpy (ctx->synth.p, synth.data(), synth.size() * sizeof (float), cudaMemcpyHostToDevice));
  return 0;
}

template<class K> int
set_smem (awm_ctx *ctx, K kernel, size_t bytes)
{
  /* the attribute sticks to the function: one driver call per kernel (and size), not one per launch */
  static std::map<std::pair<const void *, int>, size_t> done;
  size_t& have = done[{ reinterpret_cast<const void *> (kernel), ctx->device }];
  if (have >= bytes && have)
    return 0;
  CK (cudaFuncSetAttribute (kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int (bytes)));
  have = bytes;
  return 0;
}

} // namespace

void nccl_destroy (void *comm);       // defined with the awm_dist_* functions below

extern "C" {

int
awm_create (int device, awm_ctx **out)
{
  if (!out)
    return 1;
  *out = nullptr;
  int n_dev = 0;
  if (cudaGetDeviceCount (&n_dev) != cudaSuccess || n_dev <= 0)
    return 2;          // no CUDA device: the product has no CPU fallback
  if (device < 0 || device >= n_dev)
    return 3;
  awm_ctx *ctx = new awm_ctx();
  ctx->device = device;
  if (cudaSetDevice (device) != cudaSuccess || cudaStreamCreateWithFlags (&ctx->stream, cudaStreamNonBlocking) != cudaSuccess)
    {
      delete ctx;
      return 4;
    }
  if (init_tables (ctx))
    {
      fprintf (stderr, "awm_create: %s\n", ctx->err.c_str());
      delete ctx;
      return 5;
    }
  *out = ctx;
  return 0;
}

void
awm_destroy (awm_ctx *ctx)
{
  if (!ctx)
    return;
  cudaSetDevice (ctx->device);
  cudaStreamSynchronize (ctx->stream);
  DevBuf *bufs[] = { &ctx->tw, &ctx->win, &ctx->synth, &ctx->frame_mod, &ctx->pcm_own, &ctx->pcm16_own, &ctx->dbT, &ctx->have, &ctx->q, &ctx->scores, &ctx->a_ud, &ctx->a_cnt, &ctx->peaks_out, &ctx->peaks_cnt, &ctx->a_mags,
                     &ctx->cand_start, &ctx->cand_noff, &ctx->r_ud, &ctx->r_cnt, &ctx->rvalid, &ctx->r_ent_ud, &ctx->r_ent_flag, &ctx->tw1024, &ctx->vit_off, &ctx->blk_start, &ctx->D, &ctx->raw,
                     &ctx->vit_raw, &ctx->vit_types, &ctx->vit_delta, &ctx->vit_dec, &ctx->vit_bits, &ctx->vit_err, &ctx->vit_order,
                     &ctx->emb_in, &ctx->emb_out, &ctx->emb_in16, &ctx->emb_out16, &ctx->peaks, &ctx->snr, &ctx->rs_in, &ctx->rs_out, &ctx->rs_jobs, &ctx->pcm_rs,
                     &ctx->win512, &ctx->sp_clip, &ctx->sp_sub, &ctx->sp_mags, &ctx->sp_mag_jobs, &ctx->sp_cmp_jobs, &ctx->sp_best };
  for (DevBuf *b : bufs)
    b->release();
  ctx->pin.release();
  ctx->dist_send.release();
  ctx->dist_recv.release();
  if (ctx->dist_hsend) cudaFreeHost (ctx->dist_hsend);
  if (ctx->dist_hhdr) cudaFreeHost (ctx->dist_hhdr);
  if (ctx->nccl_comm)
    nccl_destroy (ctx->nccl_comm);
  for (auto& ct : ctx->coef_cache)
    ct.second.buf.release();
  for (auto& pf : ctx->pref)
    {
      pf.buf.release();
      pf.raw.release();
      if (pf.done)
        cudaEventDestroy (pf.done);
    }
  for (KeyTab& k : ctx->keys)
    {
      for (SyncTab& s : k.sync)
        {
          s.ent.release();
          s.masks.release();
          s.masks48.release();
          s.masks64.release();
          s.off.release();
          s.sorted.release();
          s.groups.release();
        }
      k.mix.release();
      k.order.release();
    }
  for (cudaEvent_t e : ctx->stage_done)
    cudaEventDestroy (e);
  if (ctx->s_in)
    cudaStreamDestroy (ctx->s_in);
  if (ctx->s_out)
    cudaStreamDestroy (ctx->s_out);
  cudaStreamDestroy (ctx->stream);
  delete ctx;
}

const char *
awm_last_error (const awm_ctx *ctx)
{
  return ctx ? ctx->err.c_str() : "no context (is a CUDA device present? there is no CPU fallback)";
}

uint64_t
awm_launch_count (const awm_ctx *ctx)
{
  return ctx ? ctx->launches : 0;
}

void *
awm_stream (awm_ctx *ctx)
{
  return ctx ? (void *) ctx->stream : nullptr;
}

int
awm_synchronize (awm_ctx *ctx)
{
  CK (cudaSetDevice (ctx->device));
  CK (cudaStreamSynchronize (ctx->stream));
  return 0;
}

void *
awm_host_alloc (size_t bytes)
{
  void *p = nullptr;
  if (cudaHostAlloc (&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess)
    {
      cudaGetLastError();
      return nullptr;
    }
  return p;
}

void
awm_host_free (void *p)
{
  if (p)
    cudaFreeHost (p);
}

int
awm_profile_enable (awm_ctx *ctx, int on)
{
  ctx->profiling = on != 0;
  return 0;
}

int
awm_profile_report (awm_ctx *ctx, char *json_out, size_t json_cap)
{
  CK (cudaSetDevice (ctx->device));
  CK (cudaStreamSynchronize (ctx->stream));
  struct Acc { std::string name; int n; double ms; double bytes; };
  std::vector<Acc> acc;
  for (auto& r : ctx->prof)
    {
      float ms = 0;
      if (r.name && cudaEventElapsedTime (&ms, r.e0, r.e1) == cudaSuccess)
        {
          bool found = false;
          for (auto& a : acc)
            if (a.name == r.name)
              {
                a.n++;
                a.ms += ms;
                a.bytes += r.bytes;
                found = true;
              }
          if (!found)
            acc.push_back ({ r.name, 1, ms, r.bytes });
        }
      cudaEventDestroy (r.e0);
      cudaEventDestroy (r.e1);
    }
  ctx->prof.clear();
  std::string js = "{";
  for (size_t i = 0; i < acc.size(); i++)
    {
      char buf[256];
      snprintf (buf, sizeof (buf), "%s\"%s\": {\"launches\": %d, \"ms\": %.6f, \"algo_bytes\": %.0f}", i ? ", " : "", acc[i].name.c_str(), acc[i].n, acc[i].ms, acc[i].bytes);
      js += buf;
    }
  js += "}";
  if (json_out && json_cap)
    {
      if (js.size() + 1 > json_cap)
        return fail (ctx, "awm_profile_report: buffer too small");
      memcpy (json_out, js.c_str(), js.size() + 1);
    }
  return 0;
}

/* ---------------------------------------------------------------- FFTProcessor */

static int
fft_batch (awm_ctx *ctx, const float *in, float *out, size_t count, int n, bool inverse)
{
  if (n != kFrame)
    return fail (ctx, "awm_fft: only n = 1024 is supported (got %d)", n);
  if (count == 0)
    return 0;
  CK (cudaSetDevice (ctx->device));
  const size_t in_elems = count * (inverse ? kFrame + 2 : kFrame), out_elems = count * (inverse ? kFrame : kFrame + 2);
  const float *d_in = in;
  float *d_out = out;
  const bool in_dev = is_device_ptr (in), out_dev = is_device_ptr (out);
  if (!in_dev)
    {
      CK (ctx->emb_in.reserve (in_elems * sizeof (float)));
      CK (cudaMemcpyAsync (ctx->emb_in.p, in, in_elems * sizeof (float), cudaMemcpyHostToDevice, ctx->stream));
      d_in = ctx->emb_in.as<float>();
    }
  if (!out_dev)
    {
      CK (ctx->emb_out.reserve (out_elems * sizeof (float)));
      d_out = ctx->emb_out.as<float>();
    }
  const size_t smem = fft_smem_bytes (kFftWarps);
  const unsigned grid = unsigned (((count + 1) / 2 + kFftWarps - 1) / kFftWarps);
  if (inverse)
    {
      if (set_smem (ctx, k_fft_c2r, smem)) return 1;
      PROF (ctx);
      k_fft_c2r<<<grid, kFftWarps * 32, smem, ctx->stream>>> (d_in, d_out, (long long) count, ctx->tw.as<float2>());
    }
  else
    {
      if (set_smem (ctx, k_fft_r2c, smem)) return 1;
      PROF (ctx);
      k_fft_r2c<<<grid, kFftWarps * 32, smem, ctx->stream>>> (d_in, d_out, (long long) count, ctx->tw.as<float2>());
    }
  LAUNCH_CHECK ("k_fft");
  if (!out_dev)
    CK (cudaMemcpyAsync (out, d_out, out_elems * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  return 0;
}

int awm_fft_r2c (awm_ctx *ctx, const float *in, float *out, size_t count, int n) { return fft_batch (ctx, in, out, count, n, false); }
int awm_fft_c2r (awm_ctx *ctx, const float *in, float *out, size_t count, int n) { return fft_batch (ctx, in, out, count, n, true); }

/* ---------------------------------------------------------------- tables */

int
awm_set_embed_tables (awm_ctx *ctx, const uint8_t *frame_mod_ab, int frames_per_block)
{
  if (!frame_mod_ab || frames_per_block <= 0)
    return fail (ctx, "awm_set_embed_tables: bad arguments");
  CK (cudaSetDevice (ctx->device));
  const size_t bytes = size_t (2) * frames_per_block * (kMaxBand + 1);
  CK (ctx->frame_mod.reserve (bytes));
  CK (cudaMemcpyAsync (ctx->frame_mod.p, frame_mod_ab, bytes, cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  ctx->embed_fpb = frames_per_block;
  return 0;
}

int
awm_set_sync_tables (awm_ctx *ctx, int key_slot, int mode, const awm_sync_entry *entries, int n_entries,
                     const int *bit_offsets, int n_bits)
{
  if (key_slot < 0 || key_slot >= AWM_MAX_KEYS || mode < 0 || mode > 1 || !entries || n_entries <= 0 || !bit_offsets || n_bits <= 0)
    return fail (ctx, "awm_set_sync_tables: bad arguments");
  if (bit_offsets[0] != 0 || bit_offsets[n_bits] != n_entries)
    return fail (ctx, "awm_set_sync_tables: bit_offsets must run from 0 to n_entries");
  for (int i = 0; i < n_entries; i++)
    for (int j = 0; j < kUD; j++)
      if (entries[i].up[j] >= kBands || entries[i].down[j] >= kBands)
        return fail (ctx, "awm_set_sync_tables: band index out of range");
  CK (cudaSetDevice (ctx->device));
  SyncTab& t = ctx->keys[key_slot].sync[mode];
  CK (t.ent.reserve (sizeof (awm_sync_entry) * n_entries));
  CK (t.off.reserve (sizeof (int) * (n_bits + 1)));
  CK (cudaMemcpyAsync (t.ent.p, entries, sizeof (awm_sync_entry) * n_entries, cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaMemcpyAsync (t.off.p, bit_offsets, sizeof (int) * (n_bits + 1), cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  if (n_bits > 6)
    return fail (ctx, "awm_set_sync_tables: at most 6 sync bits are supported");
  /* k_sync_approx walks all entries in ascending frame order (per-bit order is kept: frames are sorted inside a bit) */
  std::vector<ApproxEntry> sorted (n_entries);
  {
    std::vector<int> idx (n_entries), bit_of (n_entries);
    for (int b = 0; b < n_bits; b++)
      for (int e = bit_offsets[b]; e < bit_offsets[b + 1]; e++)
        bit_of[e] = b;
    for (int i = 0; i < n_entries; i++)
      idx[i] = i;
    std::stable_sort (idx.begin(), idx.end(), [&] (int a, int b) { return entries[a].frame < entries[b].frame; });
    for (int i = 0; i < n_entries; i++)
      {
        const awm_sync_entry& src = entries[idx[i]];
        sorted[i].frame = src.frame;
        sorted[i].bit = bit_of[idx[i]];
        sorted[i].pad = 0;
        memcpy (sorted[i].up, src.up, kUD);
        memcpy (sorted[i].down, src.down, kUD);
      }
  }
  std::vector<int> group_end;
  for (int i = 0; i < n_entries; )
    {
      int j = i;
      while (j < n_entries && j - i < 16 && sorted[j].frame - sorted[i].frame <= kApproxMaxSpan)
        j++;
      group_end.push_back (j);
      i = j;
    }
  CK (t.sorted.reserve (sorted.size() * sizeof (ApproxEntry)));
  CK (t.groups.reserve (group_end.size() * sizeof (int)));
  CK (cudaMemcpyAsync (t.sorted.p, sorted.data(), sorted.size() * sizeof (ApproxEntry), cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaMemcpyAsync (t.groups.p, group_end.data(), group_end.size() * sizeof (int), cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  {
    std::vector<unsigned char> masks, masks48, masks64;
    tc_build_masks (entries, n_entries, 128, masks);
    tc_build_masks (entries, n_entries, 48, masks48);
    tc_build_masks (entries, n_entries, 64, masks64);
    CK (t.masks.reserve (masks.size()));
    CK (t.masks48.reserve (masks48.size()));
    CK (t.masks64.reserve (masks64.size()));
    CK (cudaMemcpyAsync (t.masks.p, masks.data(), masks.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK (cudaMemcpyAsync (t.masks48.p, masks48.data(), masks48.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK (cudaMemcpyAsync (t.masks64.p, masks64.data(), masks64.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK (cudaStreamSynchronize (ctx->stream));
    t.n_chunks = int (masks.size() / tc_b_bytes (128));
    t.n_chunks48 = int (masks48.size() / tc_b_bytes (48));
    t.n_chunks64 = int (masks64.size() / tc_b_bytes (64));
  }
  t.n_groups = int (group_end.size());
  t.n_ent = n_entries;
  t.n_bits = n_bits;
  t.h_ent.assign (entries, entries + n_entries);
  t.h_off.assign (bit_offsets, bit_offsets + n_bits + 1);
  return 0;
}

int
awm_set_mix_tables (awm_ctx *ctx, int key_slot, const awm_mix_entry *entries, int n_entries,
                    const uint16_t *bit_order, int n_coded_bits, int frames_per_bit, int frames_per_block)
{
  if (key_slot < 0 || key_slot >= AWM_MAX_KEYS || !entries || !bit_order || n_coded_bits <= 0 || frames_per_bit <= 0
      || n_entries != n_coded_bits * frames_per_bit * kUD || frames_per_block <= 0)
    return fail (ctx, "awm_set_mix_tables: bad arguments");
  for (int i = 0; i < n_entries; i++)
    if (entries[i].frame >= frames_per_block || entries[i].up < kMinBand || entries[i].up > kMaxBand
        || entries[i].down < kMinBand || entries[i].down > kMaxBand)
      return fail (ctx, "awm_set_mix_tables: entry %d out of range", i);
  for (int i = 0; i < n_coded_bits; i++)
    if (bit_order[i] >= n_coded_bits)
      return fail (ctx, "awm_set_mix_tables: bit_order out of range");
  CK (cudaSetDevice (ctx->device));
  KeyTab& k = ctx->keys[key_slot];
  CK (k.mix.reserve (sizeof (awm_mix_entry) * n_entries));
  CK (k.order.reserve (sizeof (uint16_t) * n_coded_bits));
  CK (cudaMemcpyAsync (k.mix.p, entries, sizeof (awm_mix_entry) * n_entries, cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaMemcpyAsync (k.order.p, bit_order, sizeof (uint16_t) * n_coded_bits, cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  k.n_mix = n_entries;
  k.n_coded = n_coded_bits;
  k.frames_per_bit = frames_per_bit;
  k.fpb = frames_per_block;
  return 0;
}

/* ---------------------------------------------------------------- PCM */

namespace {

/* awm_pcm_bind / awm_pcm_bind_s16 / awm_pcm_bind_wav: `type` is kPcmFloat or a WavSampleType */
int
pcm_bind_any (awm_ctx *ctx, const void *pcm_v, int type, size_t n_frames, int channels, size_t pad_start, size_t pad_end)
{
  if (channels <= 0 || (!pcm_v && n_frames))
    return fail (ctx, "awm_pcm_bind: bad arguments");
  CK (cudaSetDevice (ctx->device));
  ctx->pushed = false;                           // a new bind replaces whatever awm_pcm_push_resampled saved
  const bool dev = pcm_v && is_device_ptr (pcm_v);
  awm_ctx::Prefetch *hit = nullptr;
  if (!dev && pad_start == 0 && pad_end == 0)
    for (auto& pf : ctx->pref)
      if (pf.valid && pf.src == pcm_v && pf.n_frames == n_frames && pf.ch == channels && pf.type == type)
        hit = &pf;
  if (hit)
    {
      CK (cudaStreamWaitEvent (ctx->stream, hit->done, 0));   // the prefetched copy becomes the bound PCM
      if (hit->type != kPcmFloat && wav_to_f32 (ctx, hit->type, hit->raw.p, hit->buf.as<float>(), (long long) (n_frames * channels), ctx->stream))
        return 1;
      ctx->pcm = hit->buf.as<float>();
      hit->valid = false;
    }
  else if (dev && type == kPcmFloat && pad_start == 0 && pad_end == 0)
    {
      ctx->pcm = static_cast<const float *> (pcm_v);
    }
  else
    {
      const size_t total = (pad_start + n_frames + pad_end) * channels;
      CK (ctx->pcm_own.reserve (std::max<size_t> (total, 1) * sizeof (float)));
      float *d = ctx->pcm_own.as<float>();
      if (pad_start)
        CK (cudaMemsetAsync (d, 0, pad_start * channels * sizeof (float), ctx->stream));
      if (n_frames && type == kPcmFloat)
        CK (cudaMemcpyAsync (d + pad_start * channels, pcm_v, n_frames * channels * sizeof (float),
                             dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, ctx->stream));
      if (n_frames && type != kPcmFloat)
        {
          const void *src = pcm_v;
          const size_t n_val = n_frames * channels;
          if (!dev)                                 // the stored bytes cross PCIe, they become float on the device
            {
              CK (ctx->pcm16_own.reserve (n_val * pcm_sample_bytes (type)));
              CK (cudaMemcpyAsync (ctx->pcm16_own.p, pcm_v, n_val * pcm_sample_bytes (type), cudaMemcpyHostToDevice, ctx->stream));
              src = ctx->pcm16_own.p;
            }
          if (wav_to_f32 (ctx, type, src, d + pad_start * channels, (long long) n_val, ctx->stream))
            return 1;
        }
      if (pad_end)
        CK (cudaMemsetAsync (d + (pad_start + n_frames) * channels, 0, pad_end * channels * sizeof (float), ctx->stream));
      ctx->pcm = d;
    }
  ctx->pcm_frames = pad_start + n_frames + pad_end;
  ctx->pcm_ch = channels;
  return 0;
}

/* awm_pcm_prefetch / awm_pcm_prefetch_s16 / awm_pcm_prefetch_wav.  head_frames = kFindHead: the head is found by pointer arithmetic
 * (a span that starts inside the unbound span prefetched just before it, in the same host buffer); otherwise the first head_frames
 * frames of this span are the last head_frames frames of the span prefetched just before it, and `pcm` holds the rest. */
constexpr size_t kFindHead = ~size_t (0);

int
pcm_prefetch_any (awm_ctx *ctx, const void *pcm, int type, size_t n_frames, int channels, size_t head_frames)
{
  const bool explicit_head = head_frames != kFindHead;
  if (!n_frames || channels <= 0 || (explicit_head && head_frames > n_frames) || (!pcm && (!explicit_head || head_frames < n_frames)))
    return fail (ctx, "awm_pcm_prefetch: bad arguments");
  CK (cudaSetDevice (ctx->device));
  if (pcm && is_device_ptr (pcm))
    {
      if (explicit_head && head_frames)
        return fail (ctx, "awm_pcm_prefetch: a span with a head from the previous span must be in host memory");
      return 0;                                   // nothing to do: device memory is bound in place
    }
  if (!ctx->s_in)
    {
      CK (cudaStreamCreateWithFlags (&ctx->s_in, cudaStreamNonBlocking));
      CK (cudaStreamCreateWithFlags (&ctx->s_out, cudaStreamNonBlocking));
    }
  awm_ctx::Prefetch& pf = ctx->pref[ctx->pref_next];
  awm_ctx::Prefetch& prev = ctx->pref[ctx->pref_next ^ 1];
  const size_t esz = size_t (type == kPcmFloat ? sizeof (float) : pcm_sample_bytes (type)) * size_t (channels);   // bytes per frame
  if (explicit_head && head_frames && !(prev.filled && prev.type == type && prev.ch == channels && prev.n_frames >= head_frames))
    return fail (ctx, "awm_pcm_prefetch: the previous span (%zu frames) cannot supply a head of %zu frames in this format", prev.n_frames, head_frames);
  /* the slot's previous contents may still be the bound PCM of kernels in flight: order the copy behind them */
  cudaEvent_t busy;
  CK (cudaEventCreateWithFlags (&busy, cudaEventDisableTiming));
  CK (cudaEventRecord (busy, ctx->stream));
  CK (cudaStreamWaitEvent (ctx->s_in, busy, 0));
  CK (cudaEventDestroy (busy));
  if (ctx->pcm == pf.buf.p)
    ctx->pcm_ch = 0;                              // the bound PCM is about to be overwritten: force a new bind
  const size_t n_val = n_frames * channels;
  CK (pf.buf.reserve (n_val * sizeof (float)));
  if (type != kPcmFloat)
    CK (pf.raw.reserve (n_frames * esz));
  if (!pf.done)
    CK (cudaEventCreateWithFlags (&pf.done, cudaEventDisableTiming));
  /* WAV samples stay in their stored format on the copy stream: they become float on the context stream when the span is bound
   * (pcm_bind_any), so the copy of the next span starts the moment this one has arrived */
  unsigned char *dst = static_cast<unsigned char *> (type == kPcmFloat ? pf.buf.p : pf.raw.p);
  const unsigned char *prev_bytes = static_cast<const unsigned char *> (prev.type == kPcmFloat ? prev.buf.p : prev.raw.p);
  /* Consecutive chunks of `get` overlap (WavChunkLoader: 134 s of 30 min).  The head of this span that is already on the device is
   * copied from there (device to device, ordered behind that upload on the same stream) and only the rest crosses PCIe -- 7 % fewer
   * bytes for a 1 h stream. */
  size_t head = 0;
  if (explicit_head)
    {
      head = head_frames;
      if (head)
        CK (cudaMemcpyAsync (dst, prev_bytes + (prev.n_frames - head) * esz, head * esz, cudaMemcpyDeviceToDevice, ctx->s_in));
    }
  else
    {
      const char *b0 = static_cast<const char *> (prev.src), *p0 = static_cast<const char *> (pcm);
      if (prev.valid && prev.type == type && prev.ch == channels && b0 && p0 > b0 && p0 < b0 + prev.n_frames * esz && size_t (p0 - b0) % esz == 0)
        {
          const size_t first = size_t (p0 - b0) / esz;
          head = std::min (prev.n_frames - first, n_frames);
          CK (cudaMemcpyAsync (dst, prev_bytes + first * esz, head * esz, cudaMemcpyDeviceToDevice, ctx->s_in));
        }
    }
  /* explicit head: `pcm` points at the frames after the head; found head: `pcm` is the whole span */
  const unsigned char *host = static_cast<const unsigned char *> (pcm) + (explicit_head ? 0 : head * esz);
  if (n_frames > head)
    CK (cudaMemcpyAsync (dst + head * esz, host, (n_frames - head) * esz, cudaMemcpyHostToDevice, ctx->s_in));
  CK (cudaEventRecord (pf.done, ctx->s_in));
  pf.src = pcm;
  pf.n_frames = n_frames;
  pf.ch = channels;
  pf.type = type;
  pf.valid = true;
  pf.filled = true;
  ctx->pref_next ^= 1;
  return 0;
}

} // namespace

int awm_pcm_bind (awm_ctx *ctx, const float *pcm, size_t n_frames, int channels, size_t pad_start, size_t pad_end) { return pcm_bind_any (ctx, pcm, kPcmFloat, n_frames, channels, pad_start, pad_end); }
int awm_pcm_bind_s16 (awm_ctx *ctx, const int16_t *pcm, size_t n_frames, int channels, size_t pad_start, size_t pad_end) { return pcm_bind_any (ctx, pcm, WAV_S16, n_frames, channels, pad_start, pad_end); }
int awm_pcm_prefetch (awm_ctx *ctx, const float *pcm, size_t n_frames, int channels) { return pcm_prefetch_any (ctx, pcm, kPcmFloat, n_frames, channels, kFindHead); }
int awm_pcm_prefetch_s16 (awm_ctx *ctx, const int16_t *pcm, size_t n_frames, int channels) { return pcm_prefetch_any (ctx, pcm, WAV_S16, n_frames, channels, kFindHead); }

int
awm_pcm_bind_wav (awm_ctx *ctx, const void *bytes, awm_wav_format format, size_t n_frames, int channels, size_t pad_start, size_t pad_end)
{
  const int type = wav_sample_type (format);
  if (type < 0)
    return fail (ctx, "awm_pcm_bind_wav: unsupported sample format (%d bit, %s)", format.bits, format.is_float ? "float" : "integer");
  return pcm_bind_any (ctx, bytes, type, n_frames, channels, pad_start, pad_end);
}

int
awm_pcm_prefetch_wav (awm_ctx *ctx, const void *bytes, awm_wav_format format, size_t n_frames, int channels, size_t head_frames)
{
  const int type = wav_sample_type (format);
  if (type < 0)
    return fail (ctx, "awm_pcm_prefetch_wav: unsupported sample format (%d bit, %s)", format.bits, format.is_float ? "float" : "integer");
  return pcm_prefetch_any (ctx, bytes, type, n_frames, channels, head_frames);
}

/* awm_pcm_stage / awm_pcm_stage_wait: see include/awm_b200.h */
int
awm_pcm_stage (awm_ctx *ctx, const void *pcm, int is_s16, size_t n_frames, int channels, size_t piece_frames, const float **device_out)
{
  if (!ctx || !pcm || !n_frames || channels <= 0 || !piece_frames || !device_out)
    return fail (ctx, "awm_pcm_stage: bad arguments");
  CK (cudaSetDevice (ctx->device));
  if (is_device_ptr (pcm))
    return fail (ctx, "awm_pcm_stage: the stream is already in device memory");
  if (!ctx->s_in)
    {
      CK (cudaStreamCreateWithFlags (&ctx->s_in, cudaStreamNonBlocking));
      CK (cudaStreamCreateWithFlags (&ctx->s_out, cudaStreamNonBlocking));
    }
  /* kernels in flight may still read the previous contents of the staging buffer: order the copies behind them */
  cudaEvent_t busy;
  CK (cudaEventCreateWithFlags (&busy, cudaEventDisableTiming));
  CK (cudaEventRecord (busy, ctx->stream));
  CK (cudaStreamWaitEvent (ctx->s_in, busy, 0));
  CK (cudaEventDestroy (busy));
  const size_t n_val = n_frames * channels;
  CK (ctx->staged.reserve (n_val * sizeof (float)));
  if (is_s16)
    CK (ctx->staged16.reserve (n_val * sizeof (int16_t)));
  piece_frames = (piece_frames + 1) & ~size_t (1);               // even: pieces start on 4-byte boundaries of the 16 bit copy
  const size_t n_pieces = (n_frames + piece_frames - 1) / piece_frames;
  while (ctx->stage_done.size() < n_pieces)
    {
      cudaEvent_t e;
      CK (cudaEventCreateWithFlags (&e, cudaEventDisableTiming));
      ctx->stage_done.push_back (e);
    }
  for (size_t p = 0; p < n_pieces; p++)
    {
      const size_t f0 = p * piece_frames, f1 = std::min (f0 + piece_frames, n_frames);
      const size_t v0 = f0 * channels, nv = (f1 - f0) * channels;
      if (is_s16)       /* copies only on the copy stream; a piece becomes float on the context stream when somebody waits for it */
        CK (cudaMemcpyAsync (ctx->staged16.as<int16_t>() + v0, static_cast<const int16_t *> (pcm) + v0, nv * sizeof (int16_t), cudaMemcpyHostToDevice, ctx->s_in));
      else
        CK (cudaMemcpyAsync (ctx->staged.as<float>() + v0, static_cast<const float *> (pcm) + v0, nv * sizeof (float), cudaMemcpyHostToDevice, ctx->s_in));
      CK (cudaEventRecord (ctx->stage_done[p], ctx->s_in));
    }
  ctx->stage_piece = piece_frames;
  ctx->stage_frames = n_frames;
  ctx->stage_ch = channels;
  ctx->stage_s16 = is_s16 != 0;
  ctx->stage_converted = 0;
  *device_out = ctx->staged.as<float>();
  return 0;
}

int
awm_pcm_stage_wait (awm_ctx *ctx, size_t n_frames)
{
  if (!ctx || !ctx->stage_piece || n_frames > ctx->stage_frames)
    return fail (ctx, "awm_pcm_stage_wait: nothing staged / beyond the staged stream");
  if (!n_frames)
    return 0;
  const size_t last = (n_frames - 1) / ctx->stage_piece;
  CK (cudaStreamWaitEvent (ctx->stream, ctx->stage_done[last], 0));
  for (; ctx->stage_s16 && ctx->stage_converted <= last; ctx->stage_converted++)
    {
      const size_t f0 = ctx->stage_converted * ctx->stage_piece, f1 = std::min (f0 + ctx->stage_piece, ctx->stage_frames);
      const size_t v0 = f0 * ctx->stage_ch;
      if (wav_to_f32 (ctx, WAV_S16, ctx->staged16.as<int16_t>() + v0, ctx->staged.as<float>() + v0, (long long) ((f1 - f0) * ctx->stage_ch), ctx->stream))
        return 1;
    }
  return 0;
}

/* the device copy of the bound PCM (float, [frames][channels]): lets a caller that bound 16 bit or host audio run device-pointer
 * entry points (awm_speed_scan, awm_gather) on it without another transfer */
const float *
awm_pcm_device (awm_ctx *ctx, size_t *n_frames, int *channels)
{
  if (!ctx || !ctx->pcm_ch)
    return nullptr;
  if (n_frames)
    *n_frames = ctx->pcm_frames;
  if (channels)
    *channels = ctx->pcm_ch;
  return ctx->pcm;
}

/* ---------------------------------------------------------------- embed */

namespace {

/* awm_embed / awm_embed_s16: `s16` selects 16 bit PCM buffers (in16 / out16) that are converted on the device */
int
embed_any (awm_ctx *ctx, const void *in_v, void *out_v, bool s16, size_t n_frames, int channels,
           uint64_t first_frame_number, int frames_pad_start, double water_delta,
           int limiter_block, float limiter_ceiling, double *snr_power, long long snr_pos0 = 0, long long snr_pos1 = LLONG_MAX)
{
  const float *in = s16 ? nullptr : static_cast<const float *> (in_v);
  float *out = s16 ? nullptr : static_cast<float *> (out_v);
  const int16_t *in16 = s16 ? static_cast<const int16_t *> (in_v) : nullptr;
  int16_t *out16 = s16 ? static_cast<int16_t *> (out_v) : nullptr;
  if (!ctx->embed_fpb)
    return fail (ctx, "awm_embed: awm_set_embed_tables has not been called");
  if (channels <= 0 || (n_frames && (!in_v || !out_v)))
    return fail (ctx, "awm_embed: bad arguments");
  if (snr_power)
    snr_power[0] = snr_power[1] = 0;
  if (n_frames == 0)
    return 0;
  CK (cudaSetDevice (ctx->device));
  const size_t n_val = n_frames * channels;
  /* 16 bit buffers always go through the float staging buffers; a device resident 16 bit buffer is converted in place of a copy */
  const bool in16_dev = s16 && is_device_ptr (in16), out16_dev = s16 && is_device_ptr (out16);
  const bool in_dev = !s16 && is_device_ptr (in), out_dev = !s16 && is_device_ptr (out);
  const float *d_in = in;
  float *d_out = out;
  if (!in_dev)
    {
      CK (ctx->emb_in.reserve (n_val * sizeof (float)));
      d_in = ctx->emb_in.as<float>();
    }
  if (!out_dev)
    {
      CK (ctx->emb_out.reserve (n_val * sizeof (float)));
      d_out = ctx->emb_out.as<float>();
    }
  const int16_t *d_in16 = in16;
  int16_t *d_out16 = out16;
  if (s16 && !in16_dev)
    {
      CK (ctx->emb_in16.reserve (n_val * sizeof (int16_t)));
      d_in16 = ctx->emb_in16.as<int16_t>();
    }
  if (s16 && !out16_dev)
    {
      CK (ctx->emb_out16.reserve (n_val * sizeof (int16_t)));
      d_out16 = ctx->emb_out16.as<int16_t>();
    }
  auto to_float = [&] (long long v0, long long v1, cudaStream_t st) -> int     /* values [v0, v1) of the 16 bit input -> emb_in */
    {
      if (v1 <= v0)
        return 0;
      return wav_to_f32 (ctx, WAV_S16, d_in16 + v0, ctx->emb_in.as<float>() + v0, v1 - v0, st);
    };
  auto to_s16 = [&] (long long v0, long long v1, cudaStream_t st) -> int
    {
      if (v1 <= v0)
        return 0;
      if (st == ctx->stream)
        PROF (ctx);
      k_f32_to_s16<<<unsigned (((v1 - v0 + 1) / 2 + 255) / 256), 256, 0, st>>> (d_out + v0, d_out16 + v0, v1 - v0);
      LAUNCH_CHECK ("k_f32_to_s16");
      return 0;
    };
  const long long n_real = (long long) ((n_frames + kFrame - 1) / kFrame);
  const long long n_proc = n_real + 1;
  long long n_blocks = 0;
  if (limiter_block > 0)
    {
      n_blocks = (n_proc * kFrame + limiter_block - 1) / limiter_block + 2;   // + partial first block of a mid-stream shard
      CK (ctx->peaks.reserve (n_blocks * sizeof (unsigned)));
      CK (cudaMemsetAsync (ctx->peaks.p, 0, n_blocks * sizeof (unsigned), ctx->stream));
    }
  if (snr_power)
    {
      CK (ctx->snr.reserve (2 * sizeof (double)));
      CK (cudaMemsetAsync (ctx->snr.p, 0, 2 * sizeof (double), ctx->stream));
    }
  EmbedArgs A;
  A.in = d_in;
  A.out = d_out;
  A.n_frames = (long long) n_frames;
  A.C = channels;
  A.n_proc = n_proc;
  A.fpb = ctx->embed_fpb;
  A.frame_number0 = (long long) (first_frame_number % (2ull * A.fpb)) + 2LL * A.fpb - frames_pad_start;   // WatermarkGen starts at 2*fpb - pad (src/wmadd.cc:295)
  A.frame_mod = ctx->frame_mod.as<uint8_t>();
  A.pow_up = 0.5f * float (-water_delta * 1);       // powf (mag, -Params::water_delta * data_bit_sign), src/wmadd.cc:79
  A.pow_down = 0.5f * float (-water_delta * -1);
  A.limiter_block = limiter_block;
  A.stream_pos0 = (long long) first_frame_number * kFrame;
  A.blk0 = limiter_block > 0 ? A.stream_pos0 / limiter_block : 0;
  A.peaks = ctx->peaks.as<unsigned>();
  A.snr = snr_power ? ctx->snr.as<double>() : nullptr;
  A.snr_frames = limiter_block > 0 ? n_proc : n_real;   // frames the reference loop emits (src/wmadd.cc:539-546)
  A.snr_pos0 = snr_pos0;
  A.snr_pos1 = snr_pos1;
  A.delta_only = 0;
  A.tw = ctx->tw.as<float2>();
  A.win = ctx->win.as<float>();
  A.synth = ctx->synth.as<float>();
  const size_t smem = fft_smem_bytes (kEmbedWarps) + 3 * kFrame * sizeof (float) + 2 * size_t (kEmbedWarps) * kEdge * sizeof (float2);
  if (set_smem (ctx, k_embed, smem)) return 1;
  /* stereo audio in a 16-byte aligned buffer streams through k_embed_strip (awm_embed_strip.cuh); AWM_EMBED=tile keeps k_embed */
  const char *env_embed = getenv ("AWM_EMBED");
  const bool use_strip = channels == 2 && (reinterpret_cast<uintptr_t> (A.in) & 15) == 0 && !(env_embed && !strcmp (env_embed, "tile"));
  if (use_strip)
    {
      if (!ctx->n_sms)
        CK (cudaDeviceGetAttribute (&ctx->n_sms, cudaDevAttrMultiProcessorCount, ctx->device));
      if (set_smem (ctx, k_embed_strip, kStripSmem)) return 1;
    }

  /* The buffer is processed in pieces of kPiece frames so that, for host buffers, the H2D copy of piece p+1, the
   * kernels of piece p and the D2H copy of piece p-1 overlap (three streams, events in between).  The arithmetic is
   * the same as for one launch: a piece only restricts which frames a launch emits, halo frames are read from the
   * (already copied) neighbour pieces, the limiter of a piece runs once the block peaks after it are final. */
  long long kPiece = 6144;                                   // 1024-frames per piece (6.3 M sample-frames, 25 MB of 16 bit stereo): measured best of 3072 .. 24576
  if (const char *e = getenv ("AWM_PIECE"))                  // measurement aid: other piece sizes
    kPiece = std::max (1024LL, atoll (e));
  const bool pipelined = !in_dev && !out_dev && !in16_dev && !out16_dev && n_proc > 2 * kPiece;
  const int n_pieces = pipelined ? int ((n_proc + kPiece - 1) / kPiece) : 1;
  auto piece_frames = [&] (int p, long long& fb, long long& fe) { fb = pipelined ? p * kPiece : 0; fe = pipelined ? std::min<long long> (fb + kPiece, n_proc) : n_proc; };
  auto piece_samples = [&] (int p, long long& s0, long long& s1) { long long fb, fe; piece_frames (p, fb, fe); s0 = std::min<long long> (fb * kFrame, n_frames); s1 = std::min<long long> (fe * kFrame, n_frames); };
  std::vector<cudaEvent_t> ev_in (n_pieces), ev_out (n_pieces);
  const bool trace_pipe = pipelined && getenv ("AWM_TRACE");     // device-side timeline of the three streams
  cudaEvent_t tr[4] = { nullptr, nullptr, nullptr, nullptr };
  const double t_host0 = wall_now();
  if (pipelined)
    {
      if (!ctx->s_in)
        {
          CK (cudaStreamCreateWithFlags (&ctx->s_in, cudaStreamNonBlocking));
          CK (cudaStreamCreateWithFlags (&ctx->s_out, cudaStreamNonBlocking));
        }
      for (int p = 0; p < n_pieces; p++)
        {
          CK (cudaEventCreateWithFlags (&ev_in[p], cudaEventDisableTiming));
          CK (cudaEventCreateWithFlags (&ev_out[p], cudaEventDisableTiming));
        }
      cudaEvent_t ev_start;
      CK (cudaEventCreateWithFlags (&ev_start, cudaEventDisableTiming));
      CK (cudaEventRecord (ev_start, ctx->stream));          // copies must not overtake earlier work on the context stream
      CK (cudaStreamWaitEvent (ctx->s_in, ev_start, 0));
      CK (cudaEventDestroy (ev_start));
      if (trace_pipe)
        {
          for (cudaEvent_t& e : tr)
            CK (cudaEventCreate (&e));
          CK (cudaEventRecord (tr[0], ctx->s_in));
        }
      for (int p = 0; p < n_pieces; p++)
        {
          long long s0, s1;
          piece_samples (p, s0, s1);
          if (s1 > s0 && !s16)
            CK (cudaMemcpyAsync (ctx->emb_in.as<float>() + s0 * channels, in + s0 * channels, size_t (s1 - s0) * channels * sizeof (float),
                                 cudaMemcpyHostToDevice, ctx->s_in));
          if (s1 > s0 && s16)
            {
              /* only the copy goes to the copy stream: a conversion kernel between two copies would leave the copy engine idle
               * while it runs (13 gaps per hour of audio); the conversion happens on the context stream once the piece is there */
              CK (cudaMemcpyAsync (ctx->emb_in16.as<int16_t>() + s0 * channels, in16 + s0 * channels, size_t (s1 - s0) * channels * sizeof (int16_t),
                                   cudaMemcpyHostToDevice, ctx->s_in));
            }
          CK (cudaEventRecord (ev_in[p], ctx->s_in));
        }
      if (trace_pipe)
        CK (cudaEventRecord (tr[1], ctx->s_in));
    }
  else if (s16)
    {
      if (!in16_dev)
        CK (cudaMemcpyAsync (ctx->emb_in16.p, in16, n_val * sizeof (int16_t), cudaMemcpyHostToDevice, ctx->stream));
      if (to_float (0, (long long) n_val, ctx->stream))
        return 1;
    }
  else if (!in_dev)
    CK (cudaMemcpyAsync (ctx->emb_in.p, in, n_val * sizeof (float), cudaMemcpyHostToDevice, ctx->stream));

  auto launch_limiter = [&] (int p) -> int
    {
      long long s0, s1;
      piece_samples (p, s0, s1);
      if (limiter_block > 0 && s1 > s0)
        {
          PROF (ctx);
          k_limiter<<<unsigned ((s1 - s0 + 256 * kLimiterIter - 1) / (256 * kLimiterIter)), 256, 0, ctx->stream>>> (d_out, s0, s1, channels, limiter_block, limiter_ceiling,
                                                                           ctx->peaks.as<unsigned>(), n_blocks, (long long) first_frame_number * kFrame);
          LAUNCH_CHECK ("k_limiter");
        }
      if (pipelined)
        {
          if (s1 > s0 && s16 && to_s16 (s0 * channels, s1 * channels, ctx->stream))      // the copy stream carries copies only
            return 1;
          CK (cudaEventRecord (ev_out[p], ctx->stream));
          CK (cudaStreamWaitEvent (ctx->s_out, ev_out[p], 0));
          if (s1 > s0 && !s16)
            CK (cudaMemcpyAsync (out + s0 * channels, d_out + s0 * channels, size_t (s1 - s0) * channels * sizeof (float),
                                 cudaMemcpyDeviceToHost, ctx->s_out));
          if (s1 > s0 && s16)
            CK (cudaMemcpyAsync (out16 + s0 * channels, d_out16 + s0 * channels, size_t (s1 - s0) * channels * sizeof (int16_t),
                                 cudaMemcpyDeviceToHost, ctx->s_out));
        }
      return 0;
    };
  int n_converted = 0;                                       // pieces of 16 bit input already turned into floats
  for (int p = 0; p < n_pieces; p++)
    {
      if (pipelined)
        {
          const int need = std::min (p + 1, n_pieces - 1);    // halo frame of the next piece
          CK (cudaStreamWaitEvent (ctx->stream, ev_in[need], 0));
          for (; s16 && n_converted <= need; n_converted++)
            {
              long long s0, s1;
              piece_samples (n_converted, s0, s1);
              if (to_float (s0 * channels, s1 * channels, ctx->stream))
                return 1;
            }
        }
      piece_frames (p, A.frame_begin, A.frame_end);
      if (use_strip)
        {
          /* strips long enough to make the two halo frames cheap, short enough to give every SM's warps one */
          const long long n_emit = A.frame_end - A.frame_begin;
          const int strip_len = int (std::max<long long> (16, (n_emit + (long long) ctx->n_sms * kStripWarps - 1) / ((long long) ctx->n_sms * kStripWarps)));
          const long long n_strips = (n_emit + strip_len - 1) / strip_len;
          PROF (ctx);
          k_embed_strip<<<unsigned ((n_strips + kStripWarps - 1) / kStripWarps), kStripWarps * 32, kStripSmem, ctx->stream>>> (A, strip_len);
          LAUNCH_CHECK ("k_embed_strip");
          prof_bytes (ctx, double (std::min<long long> (A.frame_end * kFrame, (long long) n_frames) - std::min<long long> (A.frame_begin * kFrame, (long long) n_frames)) * channels * 2 * sizeof (float));
          if (p > 0 && launch_limiter (p - 1))
            return 1;
          continue;
        }
      const unsigned grid = unsigned ((A.frame_end - A.frame_begin + kEmbedTile - 1) / kEmbedTile);
      PROF (ctx);
      k_embed<<<grid, kEmbedWarps * 32, smem, ctx->stream>>> (A);
      LAUNCH_CHECK ("k_embed");
      if (p > 0 && launch_limiter (p - 1))                     // peaks of the blocks after piece p-1 are final now
        return 1;
    }
  if (launch_limiter (n_pieces - 1))
    return 1;
  if (pipelined)
    {
      if (trace_pipe)
        {
          CK (cudaEventRecord (tr[2], ctx->stream));
          CK (cudaEventRecord (tr[3], ctx->s_out));
        }
      CK (cudaStreamSynchronize (ctx->s_out));
      if (trace_pipe)
        {
          float t_in = 0, t_k = 0, t_out = 0;
          cudaEventElapsedTime (&t_in, tr[0], tr[1]);
          cudaEventElapsedTime (&t_k, tr[0], tr[2]);
          cudaEventElapsedTime (&t_out, tr[0], tr[3]);
          fprintf (stderr, "[trace] embed pipeline (%d pieces): last H2D done %.2f ms, last kernel %.2f ms, last D2H %.2f ms, host issue %.2f ms\n",
                   n_pieces, t_in, t_k, t_out, (wall_now() - t_host0) * 1e3);
          for (cudaEvent_t e : tr)
            cudaEventDestroy (e);
        }
      for (int p = 0; p < n_pieces; p++)
        {
          cudaEventDestroy (ev_in[p]);
          cudaEventDestroy (ev_out[p]);
        }
    }
  else if (s16)
    {
      if (to_s16 (0, (long long) n_val, ctx->stream))
        return 1;
      if (!out16_dev)
        CK (cudaMemcpyAsync (out16, d_out16, n_val * sizeof (int16_t), cudaMemcpyDeviceToHost, ctx->stream));
    }
  else if (!out_dev)
    CK (cudaMemcpyAsync (out, d_out, n_val * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
  if (snr_power)
    CK (cudaMemcpyAsync (snr_power, ctx->snr.p, 2 * sizeof (double), cudaMemcpyDeviceToHost, ctx->stream));
  if ((s16 ? !out16_dev : !out_dev) || snr_power)
    CK (cudaStreamSynchronize (ctx->stream));
  return 0;
}

} // namespace

int
awm_embed (awm_ctx *ctx, const float *in, float *out, size_t n_frames, int channels,
           uint64_t first_frame_number, int frames_pad_start, double water_delta,
           int limiter_block, float limiter_ceiling, double *snr_power)
{
  return embed_any (ctx, in, out, false, n_frames, channels, first_frame_number, frames_pad_start, water_delta, limiter_block, limiter_ceiling, snr_power);
}

int
awm_embed_window (awm_ctx *ctx, const float *in, float *out, size_t n_frames, int channels,
                  uint64_t first_frame_number, int frames_pad_start, double water_delta,
                  int limiter_block, float limiter_ceiling, uint64_t snr_first, uint64_t snr_last, double *snr_power)
{
  return embed_any (ctx, in, out, false, n_frames, channels, first_frame_number, frames_pad_start, water_delta, limiter_block, limiter_ceiling, snr_power,
                    (long long) std::min<uint64_t> (snr_first, LLONG_MAX), (long long) std::min<uint64_t> (snr_last, LLONG_MAX));
}

int
awm_embed_s16 (awm_ctx *ctx, const int16_t *in, int16_t *out, size_t n_frames, int channels,
               uint64_t first_frame_number, int frames_pad_start, double water_delta,
               int limiter_block, float limiter_ceiling, double *snr_power)
{
  return embed_any (ctx, in, out, true, n_frames, channels, first_frame_number, frames_pad_start, water_delta, limiter_block, limiter_ceiling, snr_power);
}

/* ---------------------------------------------------------------- sync search */

int
awm_sync_approx (awm_ctx *ctx, int key_slot, int mode, uint64_t wav_first, uint64_t wav_last,
                 double water_delta, awm_search_score *scores_out, size_t max_scores, size_t *n_scores)
{
  if (key_slot < 0 || key_slot >= AWM_MAX_KEYS || mode < 0 || mode > 1 || !n_scores)
    return fail (ctx, "awm_sync_approx: bad arguments");
  SyncTab& t = ctx->keys[key_slot].sync[mode];
  const int fpb = ctx->keys[key_slot].fpb;
  if (!t.n_ent || !fpb)
    return fail (ctx, "awm_sync_approx: tables for key slot %d / mode %d not set", key_slot, mode);
  if (!ctx->pcm_ch)
    return fail (ctx, "awm_sync_approx: no PCM bound");
  CK (cudaSetDevice (ctx->device));
  const int total = fpb * (mode == AWM_MODE_CLIP ? 2 : 1);
  const long long fc = (long long) (ctx->pcm_frames / kFrame);           // frame_count (wav_data)
  const long long n_out = fc > 0 ? fc - 1 : 0;                           // sync_fft_parallel: frame_count - 1 frames per shift
  const long long n_starts = fc - total - 1 > 0 ? fc - total - 1 : 0;    // (start + total) * n_bands < fft_db.size()
  *n_scores = size_t (n_starts) * 4;
  ctx->n_scores_dev = 0;
  if (n_starts == 0)
    return 0;
  if (scores_out && max_scores < size_t (n_starts) * 4)
    return fail (ctx, "awm_sync_approx: scores_out too small (%zu < %lld)", max_scores, n_starts * 4);
  const int ld = int ((n_out + 127) / 128 * 128);
  CK (ctx->have.reserve (size_t (4) * ld));
  CK (ctx->q.reserve (size_t (n_starts) * 4 * sizeof (double)));
  CK (ctx->a_ud.reserve (size_t (n_starts) * 4 * t.n_bits * 2 * sizeof (float)));
  CK (ctx->a_cnt.reserve (size_t (n_starts) * 4 * t.n_bits * sizeof (int)));
  CK (ctx->scores.reserve (size_t (n_starts) * 4 * sizeof (awm_search_score)));
  const double norm_div = water_delta < 0.080 ? water_delta : 0.080;     // normalize_sync_quality, src/syncfinder.cc:90
  /* default: per-frame entry sums + one streaming gather (awm_approx_mags.cuh); AWM_APPROX=ring selects the kernel that walks
   * the dB matrix per start frame in the reference's exact summation order */
  static const bool force_ring = [] { const char *e = getenv ("AWM_APPROX"); return e && !strcmp (e, "ring"); } ();
  if (!force_ring && t.n_ent <= kGatherMaxEntries)
    {
      CK (ctx->a_mags.reserve (size_t (4) * t.n_ent * ld * sizeof (float2)));
      /* entry sums on the tensor cores (k_stft_mags_tc); AWM_APPROX=simt keeps them on the fp32 pipes (k_stft_mags).  Variants
       * (AWM_TC): default 12x2 = twelve FFT warps, two A buffers, mask chunks of 48 entries; 8x2 = eight FFT warps, chunks of 128
       * entries; 12x1 = twelve FFT warps, one A buffer, chunks of 128 */
      const char *env_approx = getenv ("AWM_APPROX"), *env_tc = getenv ("AWM_TC");       // read per call: tests compare the variants in one process
      const bool force_simt = env_approx && !strcmp (env_approx, "simt");
      const bool tc_12x1 = env_tc && !strcmp (env_tc, "12x1"), tc_8x2 = env_tc && !strcmp (env_tc, "8x2"), tc_11x2 = env_tc && !strcmp (env_tc, "11x2");
      if (!force_simt)
        {
          if (!ctx->n_sms)
            CK (cudaDeviceGetAttribute (&ctx->n_sms, cudaDevAttrMultiProcessorCount, ctx->device));
          const int n_tiles = 4 * int ((n_out + kTcTile - 1) / kTcTile);
          const unsigned grid = unsigned (std::min (n_tiles, ctx->n_sms));
          const char *env_tma = getenv ("AWM_TC_PCM");                      // AWM_TC_PCM=ldg: frames by global loads instead of bulk copies
          const int tma_ok = ctx->pcm_ch == 2 && (reinterpret_cast<uintptr_t> (ctx->pcm) & 15) == 0 && !(env_tma && !strcmp (env_tma, "ldg"));
#define AWM_LAUNCH_TC(FW, AB, CE, MASKS, NCH)                                                                                              \
          {                                                                                                                                 \
            const size_t smem = tc_smem_bytes<FW, AB, CE>();                                                                                \
            if (set_smem (ctx, k_stft_mags_tc<FW, AB, CE>, smem)) return 1;                                                                 \
            PROF (ctx);                                                                                                                     \
            k_stft_mags_tc<FW, AB, CE><<<grid, (FW + kTcEpiWarps + 1) * 32, smem, ctx->stream>>> (ctx->pcm, (long long) ctx->pcm_frames,    \
              ctx->pcm_ch, int (n_out), ld, MASKS.as<unsigned char>(), t.n_ent, NCH, ctx->a_mags.as<float2>(),                              \
              ctx->have.as<unsigned char>(), (long long) wav_first, (long long) wav_last, ctx->tw.as<float2>(), ctx->win.as<float>(), tma_ok); \
          }
          if (tc_12x1)
            AWM_LAUNCH_TC (12, 1, 128, t.masks, t.n_chunks)
          else if (tc_8x2)
            AWM_LAUNCH_TC (8, 2, 128, t.masks, t.n_chunks)
          else if (tc_11x2)        /* 16 warps: four per scheduler, 128 registers each (17 warps put five on one scheduler: 96 registers, spills) */
            AWM_LAUNCH_TC (11, 2, 64, t.masks64, t.n_chunks64)
          else
            AWM_LAUNCH_TC (12, 2, 48, t.masks48, t.n_chunks48)
#undef AWM_LAUNCH_TC
          LAUNCH_CHECK ("k_stft_mags_tc");
          prof_bytes (ctx, double (ctx->pcm_frames) * ctx->pcm_ch * sizeof (float) + double (4) * t.n_ent * n_out * sizeof (float2));   /* PCM in, entry sums out */
        }
      else
      {
        const size_t smem = kMagSmem2;
        if (set_smem (ctx, k_stft_mags, smem)) return 1;
        const unsigned grid = 4u * unsigned ((n_out + kMagTile - 1) / kMagTile);
        PROF (ctx);
        k_stft_mags<<<grid, kMagWarps2 * 32, smem, ctx->stream>>> (ctx->pcm, (long long) ctx->pcm_frames, ctx->pcm_ch, int (n_out), ld,
                                                                  t.ent.as<awm_sync_entry>(), t.n_ent, ctx->a_mags.as<float2>(), ctx->have.as<unsigned char>(),
                                                                  (long long) wav_first, (long long) wav_last, ctx->tw.as<float2>(), ctx->win.as<float>());
        LAUNCH_CHECK ("k_stft_mags");
        prof_bytes (ctx, double (ctx->pcm_frames) * ctx->pcm_ch * sizeof (float) + double (4) * t.n_ent * n_out * sizeof (float2));   /* PCM in, entry sums out */
      }
      dim3 grid (unsigned ((n_starts + 255) / 256), 4);
      PROF (ctx);
      if (mode == AWM_MODE_CLIP)
        k_sync_gather<true><<<grid, 256, 0, ctx->stream>>> (ctx->a_mags.as<float2>(), ctx->have.as<unsigned char>(), ld, int (n_starts), t.ent.as<awm_sync_entry>(), t.n_ent,
                                                            t.off.as<int>(), t.n_bits, ctx->a_ud.as<float>(), ctx->a_cnt.as<int>());
      else
        k_sync_gather<false><<<grid, 256, 0, ctx->stream>>> (ctx->a_mags.as<float2>(), ctx->have.as<unsigned char>(), ld, int (n_starts), t.ent.as<awm_sync_entry>(), t.n_ent,
                                                             t.off.as<int>(), t.n_bits, ctx->a_ud.as<float>(), ctx->a_cnt.as<int>());
      LAUNCH_CHECK ("k_sync_gather");
      /* every (start frame, entry) pair reads its float2 once; the per-bit sums are written once */
      prof_bytes (ctx, double (4) * n_starts * t.n_ent * sizeof (float2) + double (4) * n_starts * t.n_bits * 12.0);
    }
  else
    {
      CK (ctx->dbT.reserve (size_t (4) * kBands * ld * sizeof (float)));
      {
        const size_t smem = fft_smem_bytes (kStftWarps) + kBands * (kStftWarps + 1) * sizeof (float);
        if (set_smem (ctx, k_stft_db, smem)) return 1;
        const unsigned grid = 4u * unsigned ((n_out + kStftWarps - 1) / kStftWarps);
        PROF (ctx);
        k_stft_db<<<grid, kStftWarps * 32, smem, ctx->stream>>> (ctx->pcm, (long long) ctx->pcm_frames, ctx->pcm_ch, int (n_out), ld,
                                                                ctx->dbT.as<float>(), ctx->have.as<unsigned char>(),
                                                                (long long) wav_first, (long long) wav_last,
                                                                ctx->tw.as<float2>(), ctx->win.as<float>());
        LAUNCH_CHECK ("k_stft_db");
      }
      {
        const size_t smem = kApproxSmem;
        dim3 grid (unsigned ((n_starts + kApproxCands - 1) / kApproxCands), 4);
        if (mode == AWM_MODE_CLIP)
          {
            if (set_smem (ctx, k_sync_approx<true>, smem)) return 1;
            PROF (ctx);
            k_sync_approx<true><<<grid, kApproxThreads, smem, ctx->stream>>> (ctx->dbT.as<float>(), ctx->have.as<unsigned char>(), ld, int (n_out), int (n_starts),
                                                                            t.sorted.as<ApproxEntry>(), t.groups.as<int>(), t.n_groups, t.n_bits,
                                                                            ctx->a_ud.as<float>(), ctx->a_cnt.as<int>());
          }
        else
          {
            if (set_smem (ctx, k_sync_approx<false>, smem)) return 1;
            PROF (ctx);
            k_sync_approx<false><<<grid, kApproxThreads, smem, ctx->stream>>> (ctx->dbT.as<float>(), ctx->have.as<unsigned char>(), ld, int (n_out), int (n_starts),
                                                                             t.sorted.as<ApproxEntry>(), t.groups.as<int>(), t.n_groups, t.n_bits,
                                                                             ctx->a_ud.as<float>(), ctx->a_cnt.as<int>());
          }
        LAUNCH_CHECK ("k_sync_approx");
      }
    }
  {
    PROF (ctx);
    k_sync_quality<<<unsigned ((n_starts * 4 + 255) / 256), 256, 0, ctx->stream>>> (ctx->a_ud.as<float>(), ctx->a_cnt.as<int>(), int (n_starts), t.n_bits,
                                                                                norm_div, ctx->q.as<double>());
    LAUNCH_CHECK ("k_sync_quality");
  }
  {
    const long long n = n_starts * 4;
    PROF (ctx);
    k_local_mean<<<unsigned ((n + 255) / 256), 256, 0, ctx->stream>>> (ctx->q.as<double>(), n, ctx->scores.as<awm_search_score>());
    LAUNCH_CHECK ("k_local_mean");
  }
  ctx->n_scores_dev = size_t (n_starts) * 4;
  if (scores_out)
    {
      CK (cudaMemcpyAsync (scores_out, ctx->scores.p, size_t (n_starts) * 4 * sizeof (awm_search_score), cudaMemcpyDeviceToHost, ctx->stream));
      CK (cudaStreamSynchronize (ctx->stream));
    }
  return 0;
}

int
awm_sync_peaks (awm_ctx *ctx, double min_abs_quality, awm_search_score *out, size_t max, size_t *n)
{
  if (!n || (max && !out))
    return fail (ctx, "awm_sync_peaks: bad arguments");
  *n = 0;
  if (!ctx->n_scores_dev)
    return 0;
  CK (cudaSetDevice (ctx->device));
  /* counter and entries share one buffer ([u64 count, u64 pad][entries]) so that the usual case -- a few dozen peaks -- comes back
   * with ONE device-to-host copy and one synchronisation instead of two of each */
  constexpr size_t kHead = 16, kFirst = 2048;
  CK (ctx->peaks_out.reserve (kHead + std::max<size_t> (max, 1) * sizeof (awm_search_score)));
  unsigned char *base = ctx->peaks_out.as<unsigned char>();
  CK (cudaMemsetAsync (base, 0, kHead, ctx->stream));
  const long long ns = (long long) ctx->n_scores_dev;
  PROF (ctx);
  k_peaks<<<unsigned ((ns + 255) / 256), 256, 0, ctx->stream>>> (ctx->scores.as<awm_search_score>(), ns, min_abs_quality,
                                                                reinterpret_cast<awm_search_score *> (base + kHead), (unsigned long long) max,
                                                                reinterpret_cast<unsigned long long *> (base));
  LAUNCH_CHECK ("k_peaks");
  const size_t first = std::min (max, kFirst);
  ctx->pin.reset();
  unsigned char *stage = ctx->pin.get<unsigned char> (kHead + first * sizeof (awm_search_score));
  if (!stage)
    return fail (ctx, "awm_sync_peaks: out of page-locked memory");
  CK (cudaMemcpyAsync (stage, base, kHead + first * sizeof (awm_search_score), cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  unsigned long long cnt = 0;
  memcpy (&cnt, stage, sizeof (cnt));
  *n = size_t (cnt);
  const size_t got = std::min<size_t> (cnt, max);
  if (got)
    {
      memcpy (out, stage + kHead, std::min (got, first) * sizeof (awm_search_score));
      if (got > first)
        {
          CK (cudaMemcpyAsync (out + first, base + kHead + first * sizeof (awm_search_score), (got - first) * sizeof (awm_search_score), cudaMemcpyDeviceToHost, ctx->stream));
          CK (cudaStreamSynchronize (ctx->stream));
        }
      std::sort (out, out + got, [] (const awm_search_score& a, const awm_search_score& b) { return a.index < b.index; });
    }
  return 0;
}

/* force: -1 = default kernel choice, 0 = sliding DFT, 1 = fresh FFT per offset.  With q_out the per-offset qualities of that
 * kernel are written ([n_scores][65], invalid offsets flagged 0 in valid_out) and the scores are left alone. */
static int
refine_impl (awm_ctx *ctx, int key_slot, int mode, uint64_t wav_first, uint64_t wav_last,
             double water_delta, awm_search_score *scores, size_t n_scores, int force, double *q_out, unsigned char *valid_out)
{
  if (key_slot < 0 || key_slot >= AWM_MAX_KEYS || mode < 0 || mode > 1 || (n_scores && !scores))
    return fail (ctx, "awm_sync_refine: bad arguments");
  SyncTab& t = ctx->keys[key_slot].sync[mode];
  const int fpb = ctx->keys[key_slot].fpb;
  if (!t.n_ent || !fpb)
    return fail (ctx, "awm_sync_refine: tables for key slot %d / mode %d not set", key_slot, mode);
  if (!ctx->pcm_ch)
    return fail (ctx, "awm_sync_refine: no PCM bound");
  if (n_scores == 0)
    return 0;
  CK (cudaSetDevice (ctx->device));
  const int total = fpb * (mode == AWM_MODE_CLIP ? 2 : 1);
  const double norm_div = water_delta < 0.080 ? water_delta : 0.080;

  const size_t nc = n_scores;
  const int n_bits = t.n_bits;
  CK (ctx->cand_start.reserve (nc * sizeof (long long)));
  CK (ctx->cand_noff.reserve (nc * sizeof (int)));
  CK (ctx->r_ud.reserve (nc * kOffsets * n_bits * 2 * sizeof (float)));
  CK (ctx->r_cnt.reserve (nc * kOffsets * n_bits * sizeof (int)));
  CK (ctx->rvalid.reserve (nc * kOffsets));
  ctx->pin.reset();
  long long *h_start = ctx->pin.get<long long> (nc);
  int *h_noff = ctx->pin.get<int> (nc);
  if (!h_start || !h_noff)
    return fail (ctx, "awm_sync_refine: out of page-locked memory");
  for (size_t c = 0; c < nc; c++)
    {
      // int start = max (int (index) - sync_search_step, 0); end = index + sync_search_step; step sync_search_fine
      const long long idx = (long long) scores[c].index;
      const long long start = std::max<long long> (idx - 256, 0), end = idx + 256;
      h_start[c] = start;
      h_noff[c] = int (std::min<long long> ((end - start) / 8 + 1, kOffsets));
    }
  CK (cudaMemcpyAsync (ctx->cand_start.p, h_start, nc * sizeof (long long), cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaMemcpyAsync (ctx->cand_noff.p, h_noff, nc * sizeof (int), cudaMemcpyHostToDevice, ctx->stream));
  /* default: sliding DFT over the 65 offsets (awm_refine_slide.cuh); AWM_REFINE=fft selects the kernel that transforms every
   * frame of every offset afresh (also used for more than two channels) */
  static const bool force_fft = [] { const char *e = getenv ("AWM_REFINE"); return e && !strcmp (e, "fft"); } ();
  const bool used_slide = force < 0 ? (ctx->pcm_ch <= 2 && !force_fft) : (force == 0 && ctx->pcm_ch <= 2);
  if (used_slide)
    {
      if (!ctx->tw1024.p)
        {
          std::vector<float2> tw (1024);
          for (int p = 0; p < 1024; p++)
            {
              const double a = -2.0 * M_PI * double (p) / 1024.0;
              tw[p] = make_float2 (float (cos (a)), float (sin (a)));
            }
          CK (ctx->tw1024.reserve (tw.size() * sizeof (float2)));
          CK (cudaMemcpy (ctx->tw1024.p, tw.data(), tw.size() * sizeof (float2), cudaMemcpyHostToDevice));
        }
      const size_t n_pairs = size_t (nc) * kOffsets * t.n_ent;
      CK (ctx->r_ent_ud.reserve (n_pairs * sizeof (float2)));
      CK (ctx->r_ent_flag.reserve (n_pairs));
      const size_t smem = fft_smem_bytes (kSlideWarps);
      const long long jobs = (long long) nc * t.n_ent;
      const unsigned grid = unsigned ((jobs + kSlideWarps - 1) / kSlideWarps);
      PROF (ctx);
      if (ctx->pcm_ch == 2)
        {
          if (set_smem (ctx, k_refine_slide<2>, smem)) return 1;
          k_refine_slide<2><<<grid, kSlideWarps * 32, smem, ctx->stream>>> (ctx->pcm, (long long) ctx->pcm_frames, ctx->cand_start.as<long long>(), ctx->cand_noff.as<int>(), int (nc),
            t.ent.as<awm_sync_entry>(), t.n_ent, total, (long long) wav_first, (long long) wav_last, ctx->r_ent_ud.as<float2>(), ctx->r_ent_flag.as<unsigned char>(),
            ctx->tw.as<float2>(), ctx->tw1024.as<float2>());
        }
      else
        {
          if (set_smem (ctx, k_refine_slide<1>, smem)) return 1;
          k_refine_slide<1><<<grid, kSlideWarps * 32, smem, ctx->stream>>> (ctx->pcm, (long long) ctx->pcm_frames, ctx->cand_start.as<long long>(), ctx->cand_noff.as<int>(), int (nc),
            t.ent.as<awm_sync_entry>(), t.n_ent, total, (long long) wav_first, (long long) wav_last, ctx->r_ent_ud.as<float2>(), ctx->r_ent_flag.as<unsigned char>(),
            ctx->tw.as<float2>(), ctx->tw1024.as<float2>());
        }
      LAUNCH_CHECK ("k_refine_slide");
      /* what the kernel has to read: of every candidate's block only the SYNC frames (n_ent of the 2226), each with the 512 samples the
       * 64 slides walk over -- not the whole block */
      prof_bytes (ctx, double (nc) * double (t.n_ent) * (double (kFrame) + 512.0) * ctx->pcm_ch * sizeof (float));
      const long long n_red = (long long) nc * kOffsets * n_bits;
      PROF (ctx);
      k_refine_reduce<<<unsigned ((n_red + 127) / 128), 128, 0, ctx->stream>>> (ctx->r_ent_ud.as<float2>(), ctx->r_ent_flag.as<unsigned char>(), int (nc), t.n_ent,
        t.off.as<int>(), n_bits, ctx->cand_start.as<long long>(), ctx->cand_noff.as<int>(), (long long) ctx->pcm_frames, total,
        ctx->r_ud.as<float>(), ctx->r_cnt.as<int>(), ctx->rvalid.as<unsigned char>());
      LAUNCH_CHECK ("k_refine_reduce");
    }
  else
    {
      const size_t smem = fft_smem_bytes (kRefineWarps) + kRefineWarps * 96 * sizeof (float);
      if (set_smem (ctx, k_refine, smem)) return 1;
      const long long jobs = (long long) nc * kOffsets * n_bits;
      PROF (ctx);
      k_refine<<<unsigned ((jobs + kRefineWarps - 1) / kRefineWarps), kRefineWarps * 32, smem, ctx->stream>>> (
        ctx->pcm, (long long) ctx->pcm_frames, ctx->pcm_ch, ctx->cand_start.as<long long>(), ctx->cand_noff.as<int>(), int (nc),
        t.ent.as<awm_sync_entry>(), t.off.as<int>(), n_bits, total, (long long) wav_first, (long long) wav_last,
        ctx->r_ud.as<float>(), ctx->r_cnt.as<int>(), ctx->rvalid.as<unsigned char>(), ctx->tw.as<float2>(), ctx->win.as<float>());
      LAUNCH_CHECK ("k_refine");
      /* compulsory traffic: the sync frames of every candidate (+ the +-256 samples of the offsets) are read once -- the 65 offsets
       * x 6 bits re-read them from L2 */
      prof_bytes (ctx, double (nc) * double (t.n_ent) * (double (kFrame) + 512.0) * ctx->pcm_ch * sizeof (float));
    }
  const size_t n_ud = nc * kOffsets * n_bits * 2, n_cnt = nc * kOffsets * n_bits, n_val = nc * kOffsets;
  float *h_ud = ctx->pin.get<float> (n_ud);
  int *h_cnt = ctx->pin.get<int> (n_cnt);
  unsigned char *h_valid = ctx->pin.get<unsigned char> (n_val);
  if (!h_ud || !h_cnt || !h_valid)
    return fail (ctx, "awm_sync_refine: out of page-locked memory");
  CK (cudaMemcpyAsync (h_ud, ctx->r_ud.p, n_ud * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaMemcpyAsync (h_cnt, ctx->r_cnt.p, n_cnt * sizeof (int), cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaMemcpyAsync (h_valid, ctx->rvalid.p, n_val, cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  // sync_decode epilogue (src/syncfinder.cc:94-114,144-152) from the per-bit float sums
  auto quality_of = [&] (const float *ud, const int *cnt, size_t base) -> double
    {
      double sync_quality = 0;
      int bit_count = 0;
      for (int bit = 0; bit < n_bits; bit++)
        {
          const size_t ob = base * n_bits + bit;
          const float umag = ud[ob * 2], dmag = ud[ob * 2 + 1];
          double raw_bit;
          if (umag == 0 || dmag == 0)
            raw_bit = 0;
          else if (umag < dmag)
            raw_bit = 1 - umag / dmag;
          else
            raw_bit = dmag / umag - 1;
          sync_quality += ((bit & 1) ? raw_bit : -raw_bit) * cnt[ob];
          bit_count += cnt[ob];
        }
      if (bit_count)
        sync_quality /= bit_count;
      return sync_quality / norm_div / 2.9;
    };
  if (q_out)
    {
      for (size_t c = 0; c < nc; c++)
        for (int o = 0; o < kOffsets; o++)
          {
            const bool v = o < h_noff[c] && h_valid[c * kOffsets + o];
            valid_out[c * kOffsets + o] = v ? 1 : 0;
            q_out[c * kOffsets + o] = v ? quality_of (h_ud, h_cnt, c * kOffsets + o) : 0.0;
          }
      return 0;
    }
  if (used_slide)
    {
      /* The sliding DFT only RANKS the 65 offsets: every offset whose sliding score S lies within kVerifyMargin of the best sliding
       * score is scored again with fresh FFTs in the reference's summation order (k_refine_exact_fft / _sum compute what k_refine
       * computes), and the reference's rule picks among those exact values E.  If |S - E| <= d for all offsets, the exact arg-max o*
       * satisfies S(o*) >= E(o*) - d >= E(o') - d >= S(o') - 2d for the sliding arg-max o', so with kVerifyMargin >= 2d the exact
       * arg-max is always re-scored and index / quality are those of the exact kernel.  d is measured by
       * tests/test_gpu_stages.py::test_sync_refine_vs_oracle (asserted < kVerifyMargin / 4 on all 65 offsets of every golden candidate); neighbouring offsets
       * of a real peak differ by ~3e-3, so usually one or two offsets are re-scored. */
      constexpr double kVerifyMargin = 1e-3;
      std::vector<long long> p_start;
      std::vector<int> p_noff, p_cand, p_off;
      for (size_t c = 0; c < nc; c++)
        {
          std::vector<std::pair<double, int>> ranked;          // (-|q - local_mean|, offset): ascending sort = best first, lower offset first
          for (int o = 0; o < h_noff[c]; o++)
            if (h_valid[c * kOffsets + o])
              ranked.push_back ({ -fabs (quality_of (h_ud, h_cnt, c * kOffsets + o) - scores[c].local_mean), o });
          std::sort (ranked.begin(), ranked.end());
          size_t keep = 0;
          while (keep < ranked.size() && ranked[keep].first <= ranked[0].first + kVerifyMargin)
            keep++;
          ranked.resize (keep);
          /* the offset of the approx index itself is always re-scored: in the reference the search starts from the approx quality,
           * which there IS the exact value of that offset (same transforms, same order of additions); ours comes from the
           * entry-sum formulation and differs by ~1e-5 relative, so the exact value takes its place below */
          const int o_self = int (((long long) scores[c].index - h_start[c]) / 8);
          if (o_self < h_noff[c] && h_valid[c * kOffsets + o_self]
              && std::find_if (ranked.begin(), ranked.end(), [&] (const std::pair<double, int>& r) { return r.second == o_self; }) == ranked.end())
            ranked.push_back ({ 0.0, o_self });
          std::sort (ranked.begin(), ranked.end(), [] (const std::pair<double, int>& x, const std::pair<double, int>& y) { return x.second < y.second; });
          for (const auto& r : ranked)
            {
              p_start.push_back (h_start[c] + 8LL * r.second);
              p_noff.push_back (1);
              p_cand.push_back (int (c));
              p_off.push_back (r.second);
            }
        }
      const size_t np = p_start.size();
      float *e_ud = ctx->pin.get<float> (np * n_bits * 2);
      int *e_cnt = ctx->pin.get<int> (np * n_bits);
      unsigned char *e_valid = ctx->pin.get<unsigned char> (np);
      long long *e_start = ctx->pin.get<long long> (np);
      if (!e_ud || !e_cnt || !e_valid || !e_start)
        return fail (ctx, "awm_sync_refine: out of page-locked memory");
      std::copy (p_start.begin(), p_start.end(), e_start);
      if (np)
        {
          CK (ctx->cand_start.reserve (np * sizeof (long long)));
          CK (ctx->r_ent_ud.reserve (np * t.n_ent * 2 * kUD * sizeof (float)));
          CK (ctx->r_ud.reserve (np * n_bits * 2 * sizeof (float)));
          CK (ctx->r_cnt.reserve (np * n_bits * sizeof (int)));
          CK (ctx->rvalid.reserve (np));
          CK (cudaMemcpyAsync (ctx->cand_start.p, e_start, np * sizeof (long long), cudaMemcpyHostToDevice, ctx->stream));
          const size_t smem = fft_smem_bytes (kExactWarps) + kExactWarps * 96 * sizeof (float);
          if (set_smem (ctx, k_refine_exact_fft, smem)) return 1;
          const long long jobs = (long long) np * t.n_ent;
          PROF (ctx);
          k_refine_exact_fft<<<unsigned ((jobs + kExactWarps - 1) / kExactWarps), kExactWarps * 32, smem, ctx->stream>>> (
            ctx->pcm, (long long) ctx->pcm_frames, ctx->pcm_ch, ctx->cand_start.as<long long>(), int (np), t.ent.as<awm_sync_entry>(), t.n_ent,
            ctx->r_ent_ud.as<float>(), ctx->tw.as<float2>(), ctx->win.as<float>());
          LAUNCH_CHECK ("k_refine_exact_fft");
          /* the re-scored offsets of a candidate lie within 512 samples of each other: its sync frames are compulsory traffic once
           * (and were read by the sliding pass a moment ago: they come from L2) */
          prof_bytes (ctx, double (nc) * double (t.n_ent) * (double (kFrame) + 512.0) * ctx->pcm_ch * sizeof (float));
          PROF (ctx);
          int max_bit_frames = 1;
          for (int b = 0; b < n_bits; b++)
            max_bit_frames = std::max (max_bit_frames, t.h_off[b + 1] - t.h_off[b]);
          const size_t sum_smem = size_t (kExactSumWarps) * max_bit_frames * kUD * sizeof (float);
          if (set_smem (ctx, k_refine_exact_sum, sum_smem)) return 1;
          k_refine_exact_sum<<<unsigned ((np * n_bits * 2 + kExactSumWarps - 1) / kExactSumWarps), kExactSumWarps * 32, sum_smem, ctx->stream>>> (
            ctx->r_ent_ud.as<float>(), ctx->cand_start.as<long long>(), int (np), (long long) ctx->pcm_frames, ctx->pcm_ch, t.ent.as<awm_sync_entry>(), t.n_ent,
            t.off.as<int>(), n_bits, total, (long long) wav_first, (long long) wav_last, max_bit_frames, ctx->r_ud.as<float>(), ctx->r_cnt.as<int>(), ctx->rvalid.as<unsigned char>());
          LAUNCH_CHECK ("k_refine_exact_sum");
          CK (cudaMemcpyAsync (e_ud, ctx->r_ud.p, np * n_bits * 2 * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
          CK (cudaMemcpyAsync (e_cnt, ctx->r_cnt.p, np * n_bits * sizeof (int), cudaMemcpyDeviceToHost, ctx->stream));
          CK (cudaMemcpyAsync (e_valid, ctx->rvalid.p, np, cudaMemcpyDeviceToHost, ctx->stream));
          CK (cudaStreamSynchronize (ctx->stream));
        }
      std::vector<double> best_quality (nc);
      std::vector<uint64_t> best_index (nc);
      for (size_t c = 0; c < nc; c++)
        {
          best_quality[c] = scores[c].raw_quality;
          best_index[c] = scores[c].index;
        }
      for (size_t p = 0; p < np; p++)               // starting value: the exact quality at the approx index
        if (e_valid[p] && uint64_t (p_start[p]) == scores[p_cand[p]].index)
          best_quality[p_cand[p]] = quality_of (e_ud, e_cnt, p);
      for (size_t p = 0; p < np; p++)               // per candidate in ascending offset order
        if (e_valid[p])
          {
            const size_t c = size_t (p_cand[p]);
            const double q = quality_of (e_ud, e_cnt, p);
            if (fabs (q - scores[c].local_mean) > fabs (best_quality[c] - scores[c].local_mean))   // src/syncfinder.cc:436-440
              {
                best_quality[c] = q;
                best_index[c] = uint64_t (h_start[c] + 8LL * p_off[p]);
              }
          }
      for (size_t c = 0; c < nc; c++)
        {
          scores[c].index = best_index[c];
          scores[c].raw_quality = best_quality[c];
        }
      return 0;
    }
  for (size_t c = 0; c < nc; c++)
    {
      awm_search_score& sc = scores[c];
      double best_quality = sc.raw_quality;
      uint64_t best_index = sc.index;
      const int o_self = int (((long long) sc.index - h_start[c]) / 8);      // starting value: the exact quality at the approx index (see above)
      if (o_self < h_noff[c] && h_valid[c * kOffsets + o_self])
        best_quality = quality_of (h_ud, h_cnt, c * kOffsets + o_self);
      for (int o = 0; o < h_noff[c]; o++)
        if (h_valid[c * kOffsets + o])
          {
            const double q = quality_of (h_ud, h_cnt, c * kOffsets + o);
            if (fabs (q - sc.local_mean) > fabs (best_quality - sc.local_mean))   // src/syncfinder.cc:436-440
              {
                best_quality = q;
                best_index = uint64_t (h_start[c] + 8LL * o);
              }
          }
      sc.index = best_index;
      sc.raw_quality = best_quality;
    }
  return 0;
}

int
awm_sync_refine (awm_ctx *ctx, int key_slot, int mode, uint64_t wav_first, uint64_t wav_last,
                 double water_delta, awm_search_score *scores, size_t n_scores)
{
  return refine_impl (ctx, key_slot, mode, wav_first, wav_last, water_delta, scores, n_scores, -1, nullptr, nullptr);
}

int
awm_sync_refine_offsets (awm_ctx *ctx, int key_slot, int mode, uint64_t wav_first, uint64_t wav_last, double water_delta,
                         const awm_search_score *scores, size_t n_scores, int exact, double *quality_out, unsigned char *valid_out)
{
  if (!quality_out || !valid_out)
    return fail (ctx, "awm_sync_refine_offsets: bad arguments");
  return refine_impl (ctx, key_slot, mode, wav_first, wav_last, water_delta, const_cast<awm_search_score *> (scores), n_scores, exact ? 1 : 0,
                      quality_out, valid_out);
}

/* ---------------------------------------------------------------- multi-GPU exchange
 * NCCL is loaded on first use (dlopen), so that single-GPU users of the library do not depend on it. */
namespace {

struct NcclUniqueId { char internal[128]; };
struct NcclApi
{
  void *lib = nullptr;
  int (*GetUniqueId) (NcclUniqueId *) = nullptr;
  int (*CommInitRank) (void **, int, NcclUniqueId, int) = nullptr;
  int (*AllGather) (const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
  int (*CommDestroy) (void *) = nullptr;
  const char *(*GetErrorString) (int) = nullptr;
  std::string error;
};

NcclApi&
nccl_api()
{
  static NcclApi api;
  if (api.lib || !api.error.empty())
    return api;
  for (const char *name : { "libnccl.so.2", "libnccl.so" })
    if ((api.lib = dlopen (name, RTLD_NOW | RTLD_GLOBAL)))
      break;
  if (!api.lib)
    {
      api.error = std::string ("cannot load libnccl.so.2: ") + dlerror();
      return api;
    }
  auto sym = [&] (const char *n) { void *p = dlsym (api.lib, n); if (!p) api.error = std::string ("libnccl: missing symbol ") + n; return p; };
  api.GetUniqueId = reinterpret_cast<decltype (api.GetUniqueId)> (sym ("ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<decltype (api.CommInitRank)> (sym ("ncclCommInitRank"));
  api.AllGather = reinterpret_cast<decltype (api.AllGather)> (sym ("ncclAllGather"));
  api.CommDestroy = reinterpret_cast<decltype (api.CommDestroy)> (sym ("ncclCommDestroy"));
  api.GetErrorString = reinterpret_cast<decltype (api.GetErrorString)> (sym ("ncclGetErrorString"));
  return api;
}

} // namespace

} // extern "C"

void
nccl_destroy (void *comm)
{
  NcclApi& n = nccl_api();
  if (n.CommDestroy)
    n.CommDestroy (comm);
}

extern "C" {

int
awm_dist_unique_id (unsigned char id_out[128])
{
  NcclApi& n = nccl_api();
  if (!n.error.empty() || !id_out)
    return 1;
  NcclUniqueId id;
  if (n.GetUniqueId (&id))
    return 1;
  memcpy (id_out, id.internal, 128);
  return 0;
}

int
awm_dist_init (awm_ctx *ctx, int rank, int world, const unsigned char id[128])
{
  if (!ctx || !id || world < 1 || rank < 0 || rank >= world)
    return fail (ctx, "awm_dist_init: bad arguments");
  NcclApi& n = nccl_api();
  if (!n.error.empty())
    return fail (ctx, "awm_dist_init: %s", n.error.c_str());
  CK (cudaSetDevice (ctx->device));
  if (ctx->nccl_comm)
    {
      n.CommDestroy (ctx->nccl_comm);
      ctx->nccl_comm = nullptr;
    }
  NcclUniqueId uid;
  memcpy (uid.internal, id, 128);
  const int rc = n.CommInitRank (&ctx->nccl_comm, world, uid, rank);
  if (rc)
    return fail (ctx, "ncclCommInitRank: %s", n.GetErrorString (rc));
  ctx->dist_rank = rank;
  ctx->dist_world = world;
  return 0;
}

int
awm_dist_world (const awm_ctx *ctx, int *rank, int *world)
{
  if (!ctx)
    return 1;
  if (rank) *rank = ctx->dist_rank;
  if (world) *world = ctx->nccl_comm ? ctx->dist_world : 1;
  return 0;
}

int
awm_dist_allgather (awm_ctx *ctx, const void *send, size_t send_bytes, size_t slot_bytes, void *recv, size_t *recv_bytes)
{
  if (!ctx || (send_bytes && !send) || !recv || !recv_bytes || slot_bytes < 16 || slot_bytes % 16)
    return fail (ctx, "awm_dist_allgather: bad arguments");
  const int world = ctx->nccl_comm ? ctx->dist_world : 1;
  if (world == 1)
    {
      if (send_bytes + 8 > slot_bytes)
        return fail (ctx, "awm_dist_allgather: payload of %zu bytes does not fit a slot of %zu", send_bytes, slot_bytes);
      memcpy (recv, send, send_bytes);
      recv_bytes[0] = send_bytes;
      return 0;
    }
  NcclApi& n = nccl_api();
  CK (cudaSetDevice (ctx->device));
  CK (ctx->dist_send.reserve (slot_bytes));
  CK (ctx->dist_recv.reserve (slot_bytes * world));
  if (ctx->dist_hsend_cap < slot_bytes)
    {
      if (ctx->dist_hsend) cudaFreeHost (ctx->dist_hsend);
      if (ctx->dist_hhdr) cudaFreeHost (ctx->dist_hhdr);
      ctx->dist_hsend = ctx->dist_hhdr = nullptr;
      ctx->dist_hsend_cap = 0;
      CK (cudaMallocHost (reinterpret_cast<void **> (&ctx->dist_hsend), slot_bytes));
      CK (cudaMallocHost (reinterpret_cast<void **> (&ctx->dist_hhdr), 8 * 1024));
      ctx->dist_hsend_cap = slot_bytes;
    }
  /* slot = [u64 payload length | payload]; a payload that does not fit is announced by its length alone, every rank then sees
   * the same lengths and reports the same failure (the caller repeats the exchange with a larger slot) */
  const uint64_t len = send_bytes;
  const bool fits = send_bytes + 8 <= slot_bytes;
  memcpy (ctx->dist_hsend, &len, 8);
  if (fits && send_bytes)
    memcpy (ctx->dist_hsend + 8, send, send_bytes);
  CK (cudaMemcpyAsync (ctx->dist_send.p, ctx->dist_hsend, fits ? 8 + send_bytes : 8, cudaMemcpyHostToDevice, ctx->stream));
  const int rc = n.AllGather (ctx->dist_send.p, ctx->dist_recv.p, slot_bytes, 0 /* ncclChar */, ctx->nccl_comm, ctx->stream);
  if (rc)
    return fail (ctx, "ncclAllGather: %s", n.GetErrorString (rc));
  ctx->launches++;
  CK (cudaMemcpy2DAsync (ctx->dist_hhdr, 8, ctx->dist_recv.p, slot_bytes, 8, world, cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  bool all_fit = true;
  for (int r = 0; r < world; r++)
    {
      uint64_t l;
      memcpy (&l, ctx->dist_hhdr + 8 * r, 8);
      recv_bytes[r] = size_t (l);
      all_fit = all_fit && l + 8 <= slot_bytes;
    }
  if (!all_fit)
    return 2;                                   /* recv_bytes holds the lengths: repeat with slot_bytes >= max + 8 */
  for (int r = 0; r < world; r++)
    if (recv_bytes[r])
      CK (cudaMemcpyAsync (static_cast<unsigned char *> (recv) + size_t (r) * slot_bytes, ctx->dist_recv.as<unsigned char>() + size_t (r) * slot_bytes + 8,
                           recv_bytes[r], cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  return 0;
}

/* ---------------------------------------------------------------- block decode */

int
awm_decode_blocks (awm_ctx *ctx, int key_slot, const uint64_t *indices, size_t n_blocks, float *raw_bits_out, int *valid_out)
{
  if (key_slot < 0 || key_slot >= AWM_MAX_KEYS || (n_blocks && (!indices || !raw_bits_out || !valid_out)))
    return fail (ctx, "awm_decode_blocks: bad arguments");
  KeyTab& k = ctx->keys[key_slot];
  if (!k.n_mix)
    return fail (ctx, "awm_decode_blocks: mix tables for key slot %d not set", key_slot);
  if (!ctx->pcm_ch)
    return fail (ctx, "awm_decode_blocks: no PCM bound");
  if (n_blocks == 0)
    return 0;
  CK (cudaSetDevice (ctx->device));
  const int C = ctx->pcm_ch;
  std::vector<long long> starts;
  std::vector<size_t> which;
  for (size_t i = 0; i < n_blocks; i++)
    {
      // fft_range: empty result if samples.size() < (start_index + frame_count * frame_size) * n_channels
      const bool ok = indices[i] + uint64_t (k.fpb) * kFrame <= ctx->pcm_frames;
      valid_out[i] = ok ? 1 : 0;
      if (ok)
        {
          starts.push_back ((long long) indices[i]);
          which.push_back (i);
        }
    }
  const size_t per_blk = size_t (k.fpb) * C * kBands * sizeof (float);
  size_t batch = std::max<size_t> (1, (size_t (1) << 30) / per_blk);
  const size_t smem = fft_smem_bytes (kDecodeWarps);
  if (set_smem (ctx, k_decode_fft, smem)) return 1;
  ctx->pin.reset();
  for (size_t b0 = 0; b0 < starts.size(); b0 += batch)
    {
      const size_t nb = std::min (batch, starts.size() - b0);
      long long *h_starts = ctx->pin.get<long long> (nb);
      float *h_raw = ctx->pin.get<float> (nb * k.n_coded);
      if (!h_starts || !h_raw)
        return fail (ctx, "awm_decode_blocks: out of page-locked memory");
      std::copy (starts.begin() + b0, starts.begin() + b0 + nb, h_starts);
      CK (ctx->D.reserve (nb * per_blk));
      CK (ctx->blk_start.reserve (nb * sizeof (long long)));
      CK (ctx->raw.reserve (nb * k.n_coded * sizeof (float)));
      CK (cudaMemcpyAsync (ctx->blk_start.p, h_starts, nb * sizeof (long long), cudaMemcpyHostToDevice, ctx->stream));
      const int pairs = (C + 1) / 2;
      const long long jobs = (long long) nb * k.fpb * pairs;
      PROF (ctx);
      k_decode_fft<<<unsigned ((jobs + kDecodeWarps - 1) / kDecodeWarps), kDecodeWarps * 32, smem, ctx->stream>>> (
        ctx->pcm, (long long) ctx->pcm_frames, C, ctx->blk_start.as<long long>(), int (nb), k.fpb, ctx->D.as<float>(),
        ctx->tw.as<float2>(), ctx->win.as<float>());
      LAUNCH_CHECK ("k_decode_fft");
      prof_bytes (ctx, double (nb) * k.fpb * (double (kFrame) * C * sizeof (float) + double (C) * kBands * sizeof (float)));   /* block PCM in, band dB out */
      dim3 grid (unsigned ((k.n_coded + 127) / 128), unsigned (nb));
      PROF (ctx);
      k_mix_decode<<<grid, 128, 0, ctx->stream>>> (ctx->D.as<float>(), int (nb), C, k.fpb, k.mix.as<awm_mix_entry>(), k.frames_per_bit,
                                                   k.n_coded, k.order.as<uint16_t>(), ctx->raw.as<float>());
      LAUNCH_CHECK ("k_mix_decode");
      CK (cudaMemcpyAsync (h_raw, ctx->raw.p, nb * k.n_coded * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
      CK (cudaStreamSynchronize (ctx->stream));
      for (size_t b = 0; b < nb; b++)
        memcpy (raw_bits_out + which[b0 + b] * k.n_coded, h_raw + b * k.n_coded, k.n_coded * sizeof (float));
    }
  return 0;
}

/* ---------------------------------------------------------------- Viterbi */

int
awm_viterbi (awm_ctx *ctx, const float *raw_bits, size_t n_jobs, int n_msg_bits, const int *block_types,
             int hard, uint8_t *bits_out, float *error_out)
{
  if (n_jobs == 0)
    return 0;
  if (!raw_bits || !block_types || !bits_out || !error_out || n_msg_bits <= 0 || n_msg_bits > 4096)
    return fail (ctx, "awm_viterbi: bad arguments");
  const int steps = n_msg_bits + AWM_VITERBI_ORDER;
  std::vector<long long> off (n_jobs + 1, 0);
  for (size_t j = 0; j < n_jobs; j++)
    {
      if (block_types[j] < 0 || block_types[j] > 2)
        return fail (ctx, "awm_viterbi: bad block type %d", block_types[j]);
      off[j + 1] = off[j] + (long long) steps * (block_types[j] == AWM_BLOCK_AB ? 12 : 6);
    }
  CK (cudaSetDevice (ctx->device));
  const size_t max_jobs = 512;
  /* default: one CTA per code word (k_viterbi).  AWM_VITERBI=pair: a cluster of two CTAs per word with the metrics exchanged through
   * distributed shared memory (k_viterbi_pair, awm_viterbi_pair.cuh) -- same bits, but measured SLOWER on 110 words (1.16 vs 0.72 ms):
   * the cluster barrier of every trellis step costs ~3 us (release / acquire at cluster scope = MEMBAR.ALL.GPU in SASS) */
  const char *env_vit = getenv ("AWM_VITERBI");
  const bool use_pair = env_vit && !strcmp (env_vit, "pair");
  const size_t smem = use_pair ? viterbi_pair_smem_bytes (steps) : viterbi_smem_bytes (steps);
  if (smem > 220 * 1024)
    return fail (ctx, "awm_viterbi: %d message bits are more than the kernel holds in shared memory", n_msg_bits);
  if (use_pair ? set_smem (ctx, k_viterbi_pair, smem) : set_smem (ctx, k_viterbi, smem)) return 1;
  for (size_t j0 = 0; j0 < n_jobs; j0 += max_jobs)
    {
      const size_t nj = std::min (max_jobs, n_jobs - j0);
      const long long base = off[j0], n_raw = off[j0 + nj] - base;
      std::vector<long long> rel (nj);
      for (size_t j = 0; j < nj; j++)
        rel[j] = off[j0 + j] - base;
      CK (ctx->vit_raw.reserve (n_raw * sizeof (float)));
      CK (ctx->vit_off.reserve (nj * sizeof (long long)));
      CK (ctx->vit_types.reserve (nj * sizeof (int)));
      CK (ctx->vit_dec.reserve (nj * steps * kVitWords * sizeof (uint32_t)));
      CK (ctx->vit_bits.reserve (nj * n_msg_bits));
      CK (ctx->vit_err.reserve (nj * sizeof (float)));
      CK (ctx->vit_order.reserve (nj * sizeof (int)));
      /* host inputs / outputs pass through page-locked staging: the three uploads, the launch and the two downloads queue up
       * without the host waiting in between */
      ctx->pin.reset();
      const bool raw_on_device = is_device_ptr (raw_bits);
      float *h_in = raw_on_device ? nullptr : ctx->pin.get<float> (size_t (n_raw));
      long long *h_rel = ctx->pin.get<long long> (nj);
      int *h_types = ctx->pin.get<int> (nj);
      int *h_order = ctx->pin.get<int> (nj);
      unsigned char *h_bits = ctx->pin.get<unsigned char> (nj * n_msg_bits);
      float *h_err = ctx->pin.get<float> (nj);
      if ((!raw_on_device && !h_in) || !h_rel || !h_types || !h_order || !h_bits || !h_err)
        return fail (ctx, "awm_viterbi: out of page-locked memory");
      if (h_in)
        memcpy (h_in, raw_bits + base, size_t (n_raw) * sizeof (float));
      std::copy (rel.begin(), rel.end(), h_rel);
      std::copy (block_types + j0, block_types + j0 + nj, h_types);
      {
        /* AB words (twice the adds of an A or B word) go first in the grid, the shorter words fill the SMs they free */
        size_t k = 0;
        for (size_t j = 0; j < nj; j++)
          if (h_types[j] == AWM_BLOCK_AB)
            h_order[k++] = int (j);
        for (size_t j = 0; j < nj; j++)
          if (h_types[j] != AWM_BLOCK_AB)
            h_order[k++] = int (j);
      }
      CK (cudaMemcpyAsync (ctx->vit_raw.p, h_in ? h_in : raw_bits + base, n_raw * sizeof (float), cudaMemcpyDefault, ctx->stream));
      CK (cudaMemcpyAsync (ctx->vit_off.p, h_rel, nj * sizeof (long long), cudaMemcpyHostToDevice, ctx->stream));
      CK (cudaMemcpyAsync (ctx->vit_types.p, h_types, nj * sizeof (int), cudaMemcpyHostToDevice, ctx->stream));
      CK (cudaMemcpyAsync (ctx->vit_order.p, h_order, nj * sizeof (int), cudaMemcpyHostToDevice, ctx->stream));
      PROF (ctx);
      if (use_pair)
        k_viterbi_pair<<<unsigned (2 * nj), kVitThreads, smem, ctx->stream>>> (ctx->vit_raw.as<float>(), ctx->vit_off.as<long long>(), n_msg_bits, ctx->vit_types.as<int>(),
                                                                         hard, steps, ctx->vit_order.as<int>(), ctx->vit_dec.as<uint32_t>(),
                                                                         ctx->vit_bits.as<unsigned char>(), ctx->vit_err.as<float>());
      else
        k_viterbi<<<unsigned (nj), kVitThreads, smem, ctx->stream>>> (ctx->vit_raw.as<float>(), ctx->vit_off.as<long long>(), n_msg_bits, ctx->vit_types.as<int>(), hard,
                                                                    steps, ctx->vit_dec.as<uint32_t>(),
                                                                    ctx->vit_bits.as<unsigned char>(), ctx->vit_err.as<float>());
      LAUNCH_CHECK ("k_viterbi");
      CK (cudaMemcpyAsync (h_bits, ctx->vit_bits.p, nj * n_msg_bits, cudaMemcpyDeviceToHost, ctx->stream));
      CK (cudaMemcpyAsync (h_err, ctx->vit_err.p, nj * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
      CK (cudaStreamSynchronize (ctx->stream));
      memcpy (bits_out + j0 * n_msg_bits, h_bits, nj * n_msg_bits);
      memcpy (error_out + j0, h_err, nj * sizeof (float));
    }
  return 0;
}

} // extern "C"

/* ---------------------------------------------------------------- resampler */

namespace {

double
rs_sinc (double x)
{
  x = fabs (x);
  if (x < 1e-9)
    return 1;
  x *= M_PI;
  return sin (x) / x;
}

double
rs_window (double x)        /* three-term cosine window on [-1, 1] */
{
  x = fabs (x);
  if (x >= 1)
    return 0;
  x *= M_PI;
  return 0.384 + 0.5 * cos (x) + 0.116 * cos (2 * x);
}

/* filter table for one conversion ratio: g(d) = fc sinc (fc d) w (d / h), fc = min (1, ratio), h = ceil (hlen / fc) input
 * frames to each side; row p holds the 2h taps for a fractional position of p / 256.  Built on the host in double (a
 * few ms, cached per ratio) so that every implementation that evaluates the same formula has the same float table. */
int
coef_table (awm_ctx *ctx, double ratio, int hlen, const float **coef, int *h_out)
{
  if (!(ratio > 1.0 / 64 && ratio < 64) || hlen < 8 || hlen > 96)
    return fail (ctx, "resampler: ratio %g / hlen %d not supported", ratio, hlen);
  auto key = std::make_pair (ratio, hlen);
  auto it = ctx->coef_cache.find (key);
  if (it == ctx->coef_cache.end())
    {
      if (ctx->coef_cache.size() >= 1024)          /* data dependent ratios accumulate in long running hosts */
        {
          CK (cudaStreamSynchronize (ctx->stream));
          for (auto& ct : ctx->coef_cache)
            ct.second.buf.release();
          ctx->coef_cache.clear();
        }
      const double fc = ratio < 1 ? ratio : 1;
      const int h = int (ceil (hlen / fc));
      const int taps = 2 * h, rows = kResamplePhases + 1;
      std::vector<float> tab (size_t (rows) * taps);
      auto fill = [&] (int p0, int p1)
        {
          for (int p = p0; p < p1; p++)
            for (int j = 0; j < taps; j++)
              {
                const double d = (j - (h - 1)) - double (p) / kResamplePhases;
                tab[size_t (j) * rows + p] = float (fc * rs_sinc (fc * d) * rs_window (d / h));     /* tap major, see ResampleJob */
              }
        };
      const int n_thr = 8;
      std::vector<std::thread> thr;
      for (int t = 0; t < n_thr; t++)
        thr.emplace_back (fill, rows * t / n_thr, rows * (t + 1) / n_thr);
      for (auto& t : thr)
        t.join();
      awm_ctx::CoefTab& ct = ctx->coef_cache[key];
      ct.h = h;
      CK (ct.buf.reserve (tab.size() * sizeof (float)));
      CK (cudaMemcpy (ct.buf.p, tab.data(), tab.size() * sizeof (float), cudaMemcpyHostToDevice));
      it = ctx->coef_cache.find (key);
    }
  *coef = it->second.buf.as<float>();
  *h_out = it->second.h;
  return 0;
}

int
launch_resample (awm_ctx *ctx, const std::vector<ResampleJob>& jobs, int channels)
{
  if (jobs.empty())
    return 0;
  long long max_out = 0;
  for (const auto& j : jobs)
    max_out = std::max (max_out, j.n_out);
  if (max_out == 0)
    return 0;
  CK (ctx->rs_jobs.reserve (jobs.size() * sizeof (ResampleJob)));
  CK (cudaMemcpyAsync (ctx->rs_jobs.p, jobs.data(), jobs.size() * sizeof (ResampleJob), cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));             /* jobs is a caller-owned host vector */
  const dim3 grid (unsigned (std::min<long long> ((max_out + 255) / 256, 1 << 20)), unsigned (jobs.size()));
  PROF (ctx);
  if (channels == 2)
    k_resample<2><<<grid, 256, 0, ctx->stream>>> (ctx->rs_jobs.as<ResampleJob>(), channels);
  else if (channels == 1)
    k_resample<1><<<grid, 256, 0, ctx->stream>>> (ctx->rs_jobs.as<ResampleJob>(), channels);
  else
    k_resample<0><<<grid, 256, 0, ctx->stream>>> (ctx->rs_jobs.as<ResampleJob>(), channels);
  LAUNCH_CHECK ("k_resample");
  return 0;
}

} // namespace

int
awm_resample (awm_ctx *ctx, const float *in, size_t n_in, int channels, double ratio, int hlen, float *out, size_t n_out)
{
  if (channels <= 0 || (n_in && !in) || (n_out && !out))
    return fail (ctx, "awm_resample: bad arguments");
  if (n_out == 0)
    return 0;
  CK (cudaSetDevice (ctx->device));
  const float *coef;
  int h;
  if (coef_table (ctx, ratio, hlen, &coef, &h))
    return 1;
  const bool in_dev = n_in == 0 || is_device_ptr (in), out_dev = is_device_ptr (out);
  ResampleJob J;
  J.in = in;
  J.out = out;
  if (!in_dev)
    {
      CK (ctx->rs_in.reserve (n_in * channels * sizeof (float)));
      CK (cudaMemcpyAsync (ctx->rs_in.p, in, n_in * channels * sizeof (float), cudaMemcpyHostToDevice, ctx->stream));
      J.in = ctx->rs_in.as<float>();
    }
  if (!out_dev)
    {
      CK (ctx->rs_out.reserve (n_out * channels * sizeof (float)));
      J.out = ctx->rs_out.as<float>();
    }
  J.n_in = (long long) n_in;
  J.n_stop = J.n_in;
  J.n_out = (long long) n_out;
  J.step = 1.0 / ratio;
  J.h = h;
  J.coef = coef;
  if (launch_resample (ctx, { J }, channels))
    return 1;
  if (!out_dev)
    {
      CK (cudaMemcpyAsync (out, J.out, n_out * channels * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
      CK (cudaStreamSynchronize (ctx->stream));
    }
  return 0;
}

int
awm_pcm_push_resampled (awm_ctx *ctx, double ratio, int hlen, size_t n_out)
{
  if (!ctx->pcm_ch)
    return fail (ctx, "awm_pcm_push_resampled: no PCM bound");
  if (ctx->pushed)
    return fail (ctx, "awm_pcm_push_resampled: a resampled binding is already active");
  CK (cudaSetDevice (ctx->device));
  const float *coef;
  int h;
  if (coef_table (ctx, ratio, hlen, &coef, &h))
    return 1;
  CK (ctx->pcm_rs.reserve (std::max<size_t> (n_out, 1) * ctx->pcm_ch * sizeof (float)));
  ResampleJob J;
  J.in = ctx->pcm;
  J.out = ctx->pcm_rs.as<float>();
  J.n_in = (long long) ctx->pcm_frames;
  J.n_stop = J.n_in;
  J.n_out = (long long) n_out;
  J.step = 1.0 / ratio;
  J.h = h;
  J.coef = coef;
  if (launch_resample (ctx, { J }, ctx->pcm_ch))
    return 1;
  ctx->saved_pcm = ctx->pcm;
  ctx->saved_frames = ctx->pcm_frames;
  ctx->saved_ch = ctx->pcm_ch;
  ctx->pushed = true;
  ctx->pcm = J.out;
  ctx->pcm_frames = n_out;
  return 0;
}

int
awm_pcm_pop (awm_ctx *ctx)
{
  if (!ctx->pushed)
    return fail (ctx, "awm_pcm_pop: nothing to restore");
  ctx->pcm = ctx->saved_pcm;
  ctx->pcm_frames = ctx->saved_frames;
  ctx->pcm_ch = ctx->saved_ch;
  ctx->pushed = false;
  return 0;
}

int
awm_gather (awm_ctx *ctx, const float *src, const uint64_t *indices, size_t n, float *dst_host)
{
  if (!src || !indices || !dst_host)
    return fail (ctx, "awm_gather: bad arguments");
  if (!n)
    return 0;
  CK (cudaSetDevice (ctx->device));
  CK (ctx->rs_jobs.reserve (n * sizeof (uint64_t)));
  CK (ctx->rs_out.reserve (n * sizeof (float)));
  CK (cudaMemcpyAsync (ctx->rs_jobs.p, indices, n * sizeof (uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  PROF (ctx);
  k_gather<<<unsigned ((n + 255) / 256), 256, 0, ctx->stream>>> (src, ctx->rs_jobs.as<unsigned long long>(), (long long) n, ctx->rs_out.as<float>());
  LAUNCH_CHECK ("k_gather");
  CK (cudaMemcpyAsync (dst_host, ctx->rs_out.p, n * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  return 0;
}

int
awm_is_device_pointer (const void *p)
{
  return p && is_device_ptr (p) ? 1 : 0;
}

int
awm_copy_to_host (awm_ctx *ctx, void *dst, const void *src, size_t bytes)
{
  CK (cudaSetDevice (ctx->device));
  CK (cudaMemcpyAsync (dst, src, bytes, cudaMemcpyDefault, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  return 0;
}

/* ---------------------------------------------------------------- embed at other sample rates */

int
awm_embed_resampled (awm_ctx *ctx, const float *in, float *out, size_t n_frames, int channels, int sample_rate, int mark_sample_rate,
                     size_t n_emit, int frames_pad_start, double water_delta, int limiter_block, float limiter_ceiling, double *snr_power)
{
  if (!ctx->embed_fpb)
    return fail (ctx, "awm_embed_resampled: awm_set_embed_tables has not been called");
  if (channels <= 0 || sample_rate <= 0 || mark_sample_rate <= 0 || sample_rate == mark_sample_rate || n_emit < n_frames || (n_frames && (!in || !out)))
    return fail (ctx, "awm_embed_resampled: bad arguments");
  if (snr_power)
    snr_power[0] = snr_power[1] = 0;
  if (n_frames == 0)
    return 0;
  CK (cudaSetDevice (ctx->device));
  const double r_in = double (mark_sample_rate) / sample_rate, r_out = double (sample_rate) / mark_sample_rate;
  const float *coef_in, *coef_out;
  int h_in, h_out;
  if (coef_table (ctx, r_in, 16, &coef_in, &h_in) || coef_table (ctx, r_out, 16, &coef_out, &h_out))
    return 1;
  /* watermark frames needed for the emitted output: highest tap of output n_emit - 1 */
  const double step_out = 1.0 / r_out;
  const long long top = (long long) floor (double (n_emit - 1) * step_out) + h_out;
  const long long n_blocks44 = top / kFrame + 1;
  const long long n44 = n_blocks44 * kFrame;
  const size_t n_val = n_frames * channels;
  const bool in_dev = is_device_ptr (in), out_dev = is_device_ptr (out);
  const float *d_in = in;
  float *d_out = out;
  if (!in_dev)
    {
      CK (ctx->emb_in.reserve (n_val * sizeof (float)));
      CK (cudaMemcpyAsync (ctx->emb_in.p, in, n_val * sizeof (float), cudaMemcpyHostToDevice, ctx->stream));
      d_in = ctx->emb_in.as<float>();
    }
  if (!out_dev)
    {
      CK (ctx->emb_out.reserve (n_val * sizeof (float)));
      d_out = ctx->emb_out.as<float>();
    }
  CK (ctx->rs_in.reserve (size_t (n44) * channels * sizeof (float)));       /* x44: input at the watermark rate */
  CK (ctx->rs_out.reserve (size_t (n44) * channels * sizeof (float)));      /* wm44: watermark signal at the watermark rate */
  CK (ctx->pcm_rs.reserve (n_emit * channels * sizeof (float)));            /* watermark at the input rate */
  ctx->pushed = false;
  ctx->pcm_ch = ctx->pcm == ctx->pcm_rs.p ? 0 : ctx->pcm_ch;                 /* a pushed binding lived in pcm_rs */
  /* 1. in_resampler (src/wmadd.cc:392-393): the loop keeps feeding zero frames, so the input is zero extended */
  ResampleJob J;
  J.in = d_in; J.out = ctx->rs_in.as<float>(); J.n_in = (long long) n_frames; J.n_stop = LLONG_MAX / 4; J.n_out = n44;
  J.step = 1.0 / r_in; J.h = h_in; J.coef = coef_in;
  if (launch_resample (ctx, { J }, channels))
    return 1;
  /* 2. WatermarkGen::run on every 1024-frame of it (src/wmadd.cc:394-399) */
  {
    EmbedArgs A;
    A.in = ctx->rs_in.as<float>();
    A.out = ctx->rs_out.as<float>();
    A.n_frames = n44;
    A.C = channels;
    A.n_proc = n_blocks44 + 1;
    A.frame_begin = 0;
    A.frame_end = A.n_proc;
    A.fpb = ctx->embed_fpb;
    A.frame_number0 = 2LL * A.fpb - frames_pad_start;
    A.frame_mod = ctx->frame_mod.as<uint8_t>();
    A.pow_up = 0.5f * float (-water_delta * 1);
    A.pow_down = 0.5f * float (-water_delta * -1);
    A.limiter_block = 0;
    A.stream_pos0 = 0;
    A.blk0 = 0;
    A.peaks = nullptr;
    A.snr = nullptr;
    A.snr_frames = 0;
    A.snr_pos0 = 0;
    A.snr_pos1 = LLONG_MAX;
    A.delta_only = 1;
    A.tw = ctx->tw.as<float2>();
    A.win = ctx->win.as<float>();
    A.synth = ctx->synth.as<float>();
    const size_t smem = fft_smem_bytes (kEmbedWarps) + 3 * kFrame * sizeof (float) + 2 * size_t (kEmbedWarps) * kEdge * sizeof (float2);
    if (set_smem (ctx, k_embed, smem)) return 1;
    const unsigned grid = unsigned ((A.n_proc + kEmbedTile - 1) / kEmbedTile);
    PROF (ctx);
    k_embed<<<grid, kEmbedWarps * 32, smem, ctx->stream>>> (A);
    LAUNCH_CHECK ("k_embed");
  }
  /* 3. out_resampler (src/wmadd.cc:401-406) */
  J.in = ctx->rs_out.as<float>(); J.out = ctx->pcm_rs.as<float>(); J.n_in = n44; J.n_stop = LLONG_MAX / 4; J.n_out = (long long) n_emit;
  J.step = step_out; J.h = h_out; J.coef = coef_out;
  if (launch_resample (ctx, { J }, channels))
    return 1;
  /* 4. mix + limiter at the input rate (src/wmadd.cc:553-569) */
  long long n_lim_blocks = 0;
  if (limiter_block > 0)
    {
      n_lim_blocks = (long long) ((n_emit + limiter_block - 1) / limiter_block) + 1;
      CK (ctx->peaks.reserve (n_lim_blocks * sizeof (unsigned)));
      CK (cudaMemsetAsync (ctx->peaks.p, 0, n_lim_blocks * sizeof (unsigned), ctx->stream));
    }
  if (snr_power)
    {
      CK (ctx->snr.reserve (2 * sizeof (double)));
      CK (cudaMemsetAsync (ctx->snr.p, 0, 2 * sizeof (double), ctx->stream));
    }
  PROF (ctx);
  k_mix_peaks<<<unsigned ((n_emit + 255) / 256), 256, 0, ctx->stream>>> (d_in, (long long) n_frames, ctx->pcm_rs.as<float>(), (long long) n_emit, channels, d_out,
                                                                         limiter_block, limiter_ceiling, ctx->peaks.as<unsigned>(), snr_power ? ctx->snr.as<double>() : nullptr);
  LAUNCH_CHECK ("k_mix_peaks");
  if (limiter_block > 0)
    {
      PROF (ctx);
      k_limiter<<<unsigned ((n_frames + 256 * kLimiterIter - 1) / (256 * kLimiterIter)), 256, 0, ctx->stream>>> (d_out, 0, (long long) n_frames, channels, limiter_block, limiter_ceiling,
                                                                            ctx->peaks.as<unsigned>(), n_lim_blocks, 0);
      LAUNCH_CHECK ("k_limiter");
    }
  if (!out_dev)
    CK (cudaMemcpyAsync (out, d_out, n_val * sizeof (float), cudaMemcpyDeviceToHost, ctx->stream));
  if (snr_power)
    CK (cudaMemcpyAsync (snr_power, ctx->snr.p, 2 * sizeof (double), cudaMemcpyDeviceToHost, ctx->stream));
  if (!out_dev || snr_power)
    CK (cudaStreamSynchronize (ctx->stream));
  return 0;
}

/* ---------------------------------------------------------------- speed scan */

int
awm_speed_scan (awm_ctx *ctx, int key_slot, const float *clip, size_t clip_frames, int channels, int sample_rate,
                double seconds, const double *centers, int n_centers, const double *relative_speeds, int n_relative,
                double water_delta, double *quality_out)
{
  if (key_slot < 0 || key_slot >= AWM_MAX_KEYS || channels <= 0 || !clip || !centers || !relative_speeds || !quality_out || n_centers < 0 || n_relative < 0)
    return fail (ctx, "awm_speed_scan: bad arguments");
  SyncTab& t = ctx->keys[key_slot].sync[AWM_MODE_BLOCK];
  const int fpb = ctx->keys[key_slot].fpb;
  if (!t.n_ent || !fpb)
    return fail (ctx, "awm_speed_scan: tables for key slot %d not set", key_slot);
  if (t.n_ent > kCmpMaxEntries)
    return fail (ctx, "awm_speed_scan: %d sync entries exceed the kernel limit %d", t.n_ent, kCmpMaxEntries);
  const size_t n_jobs = size_t (n_centers) * n_relative;
  for (size_t i = 0; i < n_jobs; i++)
    quality_out[i] = 0;
  if (!n_jobs)
    return 0;
  CK (cudaSetDevice (ctx->device));
  if (!ctx->win512.p)
    {
      /* FFTAnalyzer::gen_normalized_window (sub_frame_size), src/wmcommon.cc:68-89 */
      std::vector<float> win (kSpeedFrame);
      double weight = 0;
      for (int i = 0; i < kSpeedFrame; i++)
        {
          const double w = window_cos ((i - kSpeedFrame / 2.0) / (kSpeedFrame / 2.0));
          win[i] = w;
          weight += w;
        }
      for (int i = 0; i < kSpeedFrame; i++)
        win[i] *= 2.0 / weight;
      CK (ctx->win512.reserve (win.size() * sizeof (float)));
      CK (cudaMemcpy (ctx->win512.p, win.data(), win.size() * sizeof (float), cudaMemcpyHostToDevice));
    }
  const float *d_clip = clip;
  if (!is_device_ptr (clip))
    {
      CK (ctx->sp_clip.reserve (clip_frames * channels * sizeof (float)));
      CK (cudaMemcpyAsync (ctx->sp_clip.p, clip, clip_frames * channels * sizeof (float), cudaMemcpyHostToDevice, ctx->stream));
      d_clip = ctx->sp_clip.as<float>();
    }
  /* geometry per centre: resample_ratio_truncate (in_data, center / 2, ..., seconds / center), src/wmspeed.cc:206 + src/resample.cc:100-125 */
  std::vector<ResampleJob> rj (n_centers);
  std::vector<MagJob> mj (n_centers);
  std::vector<CmpJob> cj (n_jobs);
  size_t sub_total = 0, mag_total = 0;
  int max_rows = 0;
  for (int c = 0; c < n_centers; c++)
    {
      const double ratio = centers[c] / 2;
      const float *coef;
      int h;
      if (coef_table (ctx, ratio, 16, &coef, &h))
        return 1;
      const double max_in_seconds = seconds / centers[c];
      size_t in_trunc = clip_frames;
      if (max_in_seconds > 0)
        in_trunc = std::min<size_t> (in_trunc, size_t (lrint (sample_rate * max_in_seconds)));
      const long long n_sub = lrint (double (in_trunc) * ratio);
      const int rows = n_sub > kSpeedFrame ? int ((n_sub - kSpeedFrame + kSpeedHop - 1) / kSpeedHop) : 0;
      rj[c].in = d_clip;
      rj[c].n_in = (long long) in_trunc;
      rj[c].n_stop = rj[c].n_in;
      rj[c].n_out = n_sub;
      rj[c].step = 1.0 / ratio;
      rj[c].h = h;
      rj[c].coef = coef;
      mj[c].n_sub = n_sub;
      mj[c].rows = rows;
      sub_total += size_t (n_sub) * channels;
      mag_total += size_t (rows) * t.n_ent;
      max_rows = std::max (max_rows, rows);
    }
  CK (ctx->sp_sub.reserve (std::max<size_t> (sub_total, 1) * sizeof (float)));
  CK (ctx->sp_mags.reserve (std::max<size_t> (mag_total, 1) * sizeof (float2)));
  {
    size_t so = 0, mo = 0;
    for (int c = 0; c < n_centers; c++)
      {
        rj[c].out = ctx->sp_sub.as<float>() + so;
        mj[c].sub = rj[c].out;
        mj[c].mags = ctx->sp_mags.as<float2>() + mo;
        so += size_t (rj[c].n_out) * channels;
        mo += size_t (mj[c].rows) * t.n_ent;
        for (int r = 0; r < n_relative; r++)
          {
            CmpJob& J = cj[size_t (c) * n_relative + r];
            const double rs = relative_speeds[size_t (c) * n_relative + r];
            J.mags = mj[c].mags;
            J.rows = mj[c].rows;
            J.inv = 1 / rs;                              /* relative_speed_inv, src/wmspeed.cc:274 */
            J.off_scale = (1 << 16) / rs;                /* src/wmspeed.cc:341 */
          }
      }
  }
  if (launch_resample (ctx, rj, channels))
    return 1;
  CK (ctx->sp_mag_jobs.reserve (mj.size() * sizeof (MagJob)));
  CK (ctx->sp_cmp_jobs.reserve (cj.size() * sizeof (CmpJob)));
  CK (ctx->sp_best.reserve (n_jobs * sizeof (unsigned long long)));
  CK (cudaMemcpyAsync (ctx->sp_mag_jobs.p, mj.data(), mj.size() * sizeof (MagJob), cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaMemcpyAsync (ctx->sp_cmp_jobs.p, cj.data(), cj.size() * sizeof (CmpJob), cudaMemcpyHostToDevice, ctx->stream));
  CK (cudaMemsetAsync (ctx->sp_best.p, 0, n_jobs * sizeof (unsigned long long), ctx->stream));
  if (max_rows > 0)
    {
      if (set_smem (ctx, k_speed_mags, kMagSmemBytes)) return 1;
      const dim3 grid (unsigned ((max_rows + kMagRows - 1) / kMagRows), unsigned (n_centers));
      PROF (ctx);
      k_speed_mags<<<grid, kMagWarps * 32, kMagSmemBytes, ctx->stream>>> (ctx->sp_mag_jobs.as<MagJob>(), channels, t.ent.as<awm_sync_entry>(), t.n_ent,
                                                                          ctx->tw.as<float2>(), ctx->win512.as<float>());
      LAUNCH_CHECK ("k_speed_mags");
      /* SpeedSync::compare: offsets -pad_start .. -1, pad_start = one block + one frame in search steps (src/wmspeed.cc:331) */
      const int pad_start = fpb * 4 + 4;
      const double norm_div = water_delta < 0.080 ? water_delta : 0.080;
      const dim3 cgrid (unsigned ((pad_start + 255) / 256), unsigned (n_jobs));
      PROF (ctx);
      k_speed_compare<<<cgrid, 256, 0, ctx->stream>>> (ctx->sp_cmp_jobs.as<CmpJob>(), t.ent.as<awm_sync_entry>(), t.off.as<int>(), t.n_bits, t.n_ent,
                                                       fpb, pad_start, norm_div, ctx->sp_best.as<unsigned long long>());
      LAUNCH_CHECK ("k_speed_compare");
    }
  static_assert (sizeof (double) == sizeof (unsigned long long), "quality bits");
  CK (cudaMemcpyAsync (quality_out, ctx->sp_best.p, n_jobs * sizeof (double), cudaMemcpyDeviceToHost, ctx->stream));
  CK (cudaStreamSynchronize (ctx->stream));
  return 0;
}
