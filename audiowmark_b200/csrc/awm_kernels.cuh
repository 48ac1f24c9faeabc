// awm_kernels.cuh -- sm_100a kernels of the spectral watermark hot path.
//
// Every kernel is "one warp = one 1024-point packed FFT" (awm_fft.cuh); what differs is where
// the samples come from and what is kept of the spectrum.  Reference loops replaced are cited
// per kernel (paths relative to the reference tree).
#pragma once
#include "awm_fft.cuh"
#include "awm_f32x2.cuh"
#include "../../include/awm_b200.h"
#include <math.h>

namespace awm {

// ---------------------------------------------------------------------------------------------
// shared memory carve-up common to all FFT kernels:
//   [ tw: 1024 float2 ][ win: 1024 float ][ per-warp transpose buffers ][ kernel specific ... ]
struct FftSmem
{
  float2 *tw;
  float  *win;
  float  *xbuf;       // this warp's transpose buffer
  float  *extra;      // first byte after all transpose buffers
};

constexpr size_t fft_smem_bytes (int warps) { return 1024 * sizeof (float2) + 1024 * sizeof (float) + size_t (warps) * kWarpFftSmemFloats * sizeof (float); }

__device__ __forceinline__ FftSmem
fft_smem_setup (unsigned char *smem, const float2 *g_tw, const float *g_win, int warps)
{
  FftSmem s;
  s.tw = reinterpret_cast<float2 *> (smem);
  s.win = reinterpret_cast<float *> (smem + 1024 * sizeof (float2));
  float *x0 = s.win + 1024;
  s.xbuf = x0 + (threadIdx.x >> 5) * kWarpFftSmemFloats;
  s.extra = x0 + warps * kWarpFftSmemFloats;
  for (int i = threadIdx.x; i < 1024; i += blockDim.x)
    {
      s.tw[i] = g_tw[i];
      s.win[i] = g_win ? g_win[i] : 1.0f;
    }
  __syncthreads();
  return s;
}

// load (and window) one pair of real sequences: re <- channel chA, im <- channel chB (or 0)
// from interleaved PCM, sample-frames [start, start+1024), zero beyond n_frames.
__device__ __forceinline__ void
load_pair (const float *__restrict__ pcm, long long n_frames, int C, long long start, int chA, int chB,
           const float *win, float (&re)[32], float (&im)[32], int lane)
{
  if (C == 2 && chB == 1 && start >= 0 && start + kFrame <= n_frames)
    {
      /* common case: whole stereo frame inside the buffer -> one base pointer, immediate offsets, no bounds tests */
      const float2 *p = reinterpret_cast<const float2 *> (pcm) + start + lane;
#pragma unroll
      for (int j = 0; j < 32; j++)
        {
          const float2 v = __ldg (p + 32 * j);
          const float w = win[32 * j + lane];
          re[j] = __fmul_rn (v.x, w);            /* spelled out: not to be fused into the first butterfly */
          im[j] = __fmul_rn (v.y, w);
        }
    }
  else if (C == 2 && chB == 1)
    {
      const float2 *p2 = reinterpret_cast<const float2 *> (pcm);
#pragma unroll
      for (int j = 0; j < 32; j++)
        {
          const int n = 32 * j + lane;
          const long long pos = start + n;
          float2 v = make_float2 (0.f, 0.f);
          if (pos >= 0 && pos < n_frames)
            v = __ldg (p2 + pos);
          const float w = win[n];
          re[j] = __fmul_rn (v.x, w);            /* spelled out: not to be fused into the first butterfly */
          im[j] = __fmul_rn (v.y, w);
        }
    }
  else
    {
#pragma unroll
      for (int j = 0; j < 32; j++)
        {
          const int n = 32 * j + lane;
          const long long pos = start + n;
          float a = 0.f, b = 0.f;
          if (pos >= 0 && pos < n_frames)
            {
              a = __ldg (pcm + pos * C + chA);
              if (chB >= 0)
                b = __ldg (pcm + pos * C + chB);
            }
          const float w = win[n];
          re[j] = __fmul_rn (a, w);
          im[j] = __fmul_rn (b, w);
        }
    }
}

// channel-summed band dB of one frame (SyncFinder::sync_fft inner loop, src/syncfinder.cc:590-598):
// acc[K2] of lane k1 is the band value for bin k1 + 32*K2 (valid where 20 <= bin <= 100).
__device__ __forceinline__ void
frame_db_sum (const float *__restrict__ pcm, long long n_frames, int C, long long start,
              const FftSmem& s, int lane, float (&acc)[4])
{
  acc[0] = acc[1] = acc[2] = acc[3] = 0.f;
  for (int chA = 0; chA < C; chA += 2)
    {
      const int chB = (chA + 1 < C) ? chA + 1 : -1;
      float re[32], im[32];
      load_pair (pcm, n_frames, C, start, chA, chB, s.win, re, im, lane);
      const unsigned zero = pair_zero_mask (re, im);
      fft1024_warp (re, im, s.tw, s.xbuf, lane);
      float ar, ai, br, bi;
      unpack_pair<0> (re, im, lane, ar, ai, br, bi, zero);
      acc[0] += db_from_complex (ar, ai, -96.f);
      if (chB >= 0) acc[0] += db_from_complex (br, bi, -96.f);
      unpack_pair<1> (re, im, lane, ar, ai, br, bi, zero);
      acc[1] += db_from_complex (ar, ai, -96.f);
      if (chB >= 0) acc[1] += db_from_complex (br, bi, -96.f);
      unpack_pair<2> (re, im, lane, ar, ai, br, bi, zero);
      acc[2] += db_from_complex (ar, ai, -96.f);
      if (chB >= 0) acc[2] += db_from_complex (br, bi, -96.f);
      unpack_pair<3> (re, im, lane, ar, ai, br, bi, zero);
      acc[3] += db_from_complex (ar, ai, -96.f);
      if (chB >= 0) acc[3] += db_from_complex (br, bi, -96.f);
    }
}

// scatter the (up to 4) band values a lane holds into a dense 81-entry array
__device__ __forceinline__ void
bands_to_array (const float (&acc)[4], int lane, float *dst, int stride)
{
#pragma unroll
  for (int k2 = 0; k2 < 4; k2++)
    {
      const int band = lane + 32 * k2 - kMinBand;
      if (band >= 0 && band < kBands)
        dst[band * stride] = acc[k2];
    }
}

// =============================================================================================
// FFTProcessor::fft / ifft, batched (src/fft.cc:82-118).  One warp = two consecutive transforms.
// =============================================================================================
constexpr int kFftWarps = 8;

__global__ void __launch_bounds__ (kFftWarps * 32)
k_fft_r2c (const float *__restrict__ in, float *__restrict__ out, long long count, const float2 *g_tw)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, g_tw, nullptr, kFftWarps);
  const int lane = threadIdx.x & 31;
  const long long p = (long long) blockIdx.x * kFftWarps + (threadIdx.x >> 5);
  if (2 * p >= count)
    return;
  const bool have_b = 2 * p + 1 < count;
  const float *a = in + 2 * p * kFrame, *b = a + kFrame;
  float re[32], im[32];
#pragma unroll
  for (int j = 0; j < 32; j++)
    {
      re[j] = a[32 * j + lane];
      im[j] = have_b ? b[32 * j + lane] : 0.f;
    }
  const unsigned zero = pair_zero_mask (re, im);
  fft1024_warp (re, im, s.tw, s.xbuf, lane);
  float2 *oa = reinterpret_cast<float2 *> (out + 2 * p * (kFrame + 2)), *ob = oa + (kFrame / 2 + 1);
  auto emit = [&] (int k, bool pred, float ar, float ai, float br, float bi)
    {
      if (pred)
        {
          oa[k] = make_float2 (ar, ai);
          if (have_b)
            ob[k] = make_float2 (br, bi);
        }
    };
  float ar, ai, br, bi;
#define AWM_EMIT(K2) unpack_pair<K2> (re, im, lane, ar, ai, br, bi, zero); emit (lane + 32 * K2, true, ar, ai, br, bi);
  AWM_EMIT (0) AWM_EMIT (1) AWM_EMIT (2) AWM_EMIT (3) AWM_EMIT (4) AWM_EMIT (5) AWM_EMIT (6) AWM_EMIT (7)
  AWM_EMIT (8) AWM_EMIT (9) AWM_EMIT (10) AWM_EMIT (11) AWM_EMIT (12) AWM_EMIT (13) AWM_EMIT (14) AWM_EMIT (15)
#undef AWM_EMIT
  unpack_pair<16> (re, im, lane, ar, ai, br, bi, zero);
  emit (512, lane == 0, ar, ai, br, bi);
}

__global__ void __launch_bounds__ (kFftWarps * 32)
k_fft_c2r (const float *__restrict__ in, float *__restrict__ out, long long count, const float2 *g_tw)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, g_tw, nullptr, kFftWarps);
  const int lane = threadIdx.x & 31;
  const long long p = (long long) blockIdx.x * kFftWarps + (threadIdx.x >> 5);
  if (2 * p >= count)
    return;
  const bool have_b = 2 * p + 1 < count;
  const float2 *A = reinterpret_cast<const float2 *> (in + 2 * p * (kFrame + 2)), *B = A + (kFrame / 2 + 1);
  float re[32], im[32];
  // D[k] = A[k] + i B[k] (k <= 512), D[k] = conj A[N-k] + i conj B[N-k] (k > 512); inverse = swap (FFT (swap D))
#pragma unroll
  for (int j = 0; j < 32; j++)
    {
      const int k = 32 * j + lane;
      const int ks = k <= 512 ? k : kFrame - k;
      float2 a = A[ks], b = have_b ? B[ks] : make_float2 (0.f, 0.f);
      if (ks == 0 || ks == 512)     // c2r ignores the imaginary part of DC / Nyquist
        a.y = b.y = 0.f;
      if (k > 512)
        {
          a.y = -a.y;
          b.y = -b.y;
        }
      const float dr = a.x - b.y, di = a.y + b.x;
      re[j] = di;
      im[j] = dr;
    }
  fft1024_warp (re, im, s.tw, s.xbuf, lane);
  float *oa = out + 2 * p * kFrame, *ob = oa + kFrame;
#pragma unroll
  for (int i = 0; i < 32; i++)
    {
      const int n = lane + 32 * brev5 (i);
      oa[n] = im[i];
      if (have_b)
        ob[n] = re[i];
    }
}

// =============================================================================================
// SyncFinder::sync_fft / sync_fft_parallel for all four 256-sample shifts
// (src/syncfinder.cc:560-657): db[shift][band][frame] (band-major so the per-candidate gathers of
// k_sync_approx are coalesced over consecutive start frames) and have[shift][frame].
// grid = 4 * ceil(n_out/8) CTAs (shift = blockIdx.x & 3), 8 warps, warp = one frame.
// =============================================================================================
constexpr int kStftWarps = 8;

__global__ void __launch_bounds__ (kStftWarps * 32, 2)
k_stft_db (const float *__restrict__ pcm, long long n_frames, int C, int n_out, int ld,
           float *__restrict__ dbT, unsigned char *__restrict__ have,
           long long wav_first, long long wav_last, const float2 *g_tw, const float *g_win)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, g_tw, g_win, kStftWarps);
  float *tile = s.extra;                               // [81][kStftWarps + 1]
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  // the four shifts of a frame tile are neighbouring CTAs, so the tile's samples are fetched from HBM once (L2 serves the rest)
  const int shift_idx = blockIdx.x & 3, tile_idx = blockIdx.x >> 2;
  const int f = tile_idx * kStftWarps + w;
  const long long start = (long long) shift_idx * 256 + (long long) f * kFrame;

  bool ok = f < n_out;
  if (ok)
    {
      const long long f_first = start * C, f_last = (start + kFrame) * C;
      if (f_last < wav_first || f_first > wav_last)   // frame in leading / trailing digital silence
        ok = false;
    }
  float acc[4] = { 0.f, 0.f, 0.f, 0.f };
  if (ok)
    frame_db_sum (pcm, n_frames, C, start, s, lane, acc);
  bands_to_array (acc, lane, tile + w, kStftWarps + 1);
  if (lane == 0 && f < n_out)
    have[(size_t) shift_idx * ld + f] = ok ? 1 : 0;
  __syncthreads();
  for (int i = threadIdx.x; i < kBands * kStftWarps; i += blockDim.x)
    {
      const int band = i / kStftWarps, ww = i % kStftWarps;
      const int ff = tile_idx * kStftWarps + ww;
      if (ff < n_out)
        dbT[((size_t) shift_idx * kBands + band) * ld + ff] = tile[band * (kStftWarps + 1) + ww];
    }
}

// =============================================================================================
// SyncFinder::sync_decode for every start frame (src/syncfinder.cc:116-153, bit_quality :94-114,
// normalize_sync_quality :80-91).  One thread = one candidate start frame, float sums in the reference's
// order (per sync bit: frames ascending, 30 up / 30 down bands each).
//
// A CTA owns kApproxCands consecutive start frames of one shift.  Candidate s reads db[band][s + frame(e)] for
// each sync entry e, so while the entries are walked in ascending frame order the CTA's working set is a
// sliding window of the band-major dB matrix: it is staged in a shared-memory ring (81 bands x kApproxRing
// frames) that is topped up group by group, and every dB value is fetched from L2 once per CTA instead of
// once per (candidate, entry) -- 30600 float adds per candidate then run at shared-memory speed.
//   ent_sorted: all entries of all bits merged by ascending frame (per-bit order is preserved),
//               64 bytes each: u16 frame, u8 bit, u8 pad, u8 up[30], u8 down[30]
//   group_end : entries [group_end[g-1], group_end[g]) span at most kApproxMaxSpan frames
// out[s*4 + shift] so that the array is already sorted by index = s*1024 + shift*256.
// =============================================================================================
constexpr int kApproxCands = 256;          // candidates per CTA
constexpr int kApproxSplit = 3;            // thread groups per candidate: group j sums sync bits 2j, 2j+1 (more warps to hide latency)
constexpr int kApproxThreads = kApproxCands * kApproxSplit;
constexpr int kApproxRing = 512;           // ring length in frames (power of two)
constexpr int kApproxMaxSpan = (kApproxRing - kApproxCands) / 2 - 1;   // two consecutive groups fit the ring: group g+1 is prefetched while g is summed
struct ApproxEntry { uint16_t frame; uint8_t bit, pad; uint8_t up[30], down[30]; };
static_assert (sizeof (ApproxEntry) == 64, "ApproxEntry must be 64 bytes");
constexpr size_t kApproxSmem = size_t (kBands) * kApproxRing * sizeof (float) + kApproxRing;

template<bool CHECK_HAVE> __global__ void __launch_bounds__ (kApproxThreads, 1)
k_sync_approx (const float *__restrict__ dbT, const unsigned char *__restrict__ have, int ld, int n_out, int n_starts,
               const ApproxEntry *__restrict__ ent_sorted, const int *__restrict__ group_end, int n_groups, int n_bits,
               float *__restrict__ out_ud /* [4][n_starts][n_bits][2] */, int *__restrict__ out_cnt /* [4][n_starts][n_bits] */)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  float *ring = reinterpret_cast<float *> (smem);                         // [band][kApproxRing]
  unsigned char *hring = smem + size_t (kBands) * kApproxRing * sizeof (float);   // have flags, same slots
  const int shift_idx = blockIdx.y;
  const int s0 = blockIdx.x * kApproxCands;
  const int cand = threadIdx.x % kApproxCands, part = threadIdx.x / kApproxCands;   // part is warp-uniform
  const int s = s0 + cand;
  const float *db = dbT + (size_t) shift_idx * kBands * ld;
  const unsigned char *hv = have + (size_t) shift_idx * ld;

  float u0 = 0, u1 = 0, d0 = 0, d1 = 0;                                   // sums of sync bits 2*part and 2*part + 1
  int c0 = 0, c1 = 0;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int loaded = s0;                                                          // frames < loaded are (or were) in the ring
  // asynchronous top-up of the ring with the frames group g needs (cp.async: no registers, no stall until the wait)
  auto prefetch = [&] (int g)
    {
      const int e_first = g ? group_end[g - 1] : 0;
      const int fr_first = ent_sorted[e_first].frame, fr_last = ent_sorted[group_end[g] - 1].frame;
      const int need_lo = max (loaded, s0 + fr_first), need_hi = s0 + fr_last + kApproxCands;
      for (int band = warp; band < kBands; band += kApproxThreads / 32)
        {
          const float *src = db + (size_t) band * ld;
          float *dst = ring + band * kApproxRing;
          for (int f = need_lo + lane; f < need_hi; f += 32)
            {
              if (f < n_out)
                {
                  const unsigned sa = (unsigned) __cvta_generic_to_shared (dst + (f & (kApproxRing - 1)));
                  asm volatile ("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(sa), "l"(src + f) : "memory");
                }
              else
                dst[f & (kApproxRing - 1)] = 0.f;
            }
        }
      if (CHECK_HAVE)
        for (int f = need_lo + threadIdx.x; f < need_hi; f += kApproxThreads)
          hring[f & (kApproxRing - 1)] = f < n_out ? hv[f] : 0;
      loaded = need_hi;
    };
  prefetch (0);
  asm volatile ("cp.async.wait_all;" ::: "memory");
  __syncthreads();
  int e = 0;
  for (int g = 0; g < n_groups; g++)
    {
      const int e_end = group_end[g];
      // group g+1 may be fetched while g is summed if both fit the ring together (normally true: groups span <= kApproxMaxSpan)
      bool early = false;
      if (g + 1 < n_groups)
        {
          early = int (ent_sorted[group_end[g + 1] - 1].frame) - int (ent_sorted[e].frame) + kApproxCands < kApproxRing;
          if (early)
            prefetch (g + 1);
        }
      for (; e < e_end; e++)
        {
          const uint4 *e4 = reinterpret_cast<const uint4 *> (ent_sorted + e);
          const uint4 w0 = __ldg (e4), w1 = __ldg (e4 + 1), w2 = __ldg (e4 + 2), w3 = __ldg (e4 + 3);
          const unsigned words[16] = { w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w, w2.x, w2.y, w2.z, w2.w, w3.x, w3.y, w3.z, w3.w };
          const int frame = words[0] & 0xffff, bit = (words[0] >> 16) & 0xff;
          if ((bit >> 1) != part)
            continue;                                                       // another thread group owns this sync bit
          const int slot = (s + frame) & (kApproxRing - 1);
          if (CHECK_HAVE && !hring[slot])
            continue;
          const float *base = ring + slot;
          const bool odd = bit & 1;
          float um = odd ? u1 : u0, dm = odd ? d1 : d0;
#pragma unroll
          for (int i = 0; i < kUD; i++)
            {
              const unsigned ub = (words[(4 + i) >> 2] >> (8 * ((4 + i) & 3))) & 0xffu;
              const unsigned dbn = (words[(34 + i) >> 2] >> (8 * ((34 + i) & 3))) & 0xffu;
              um += base[ub * kApproxRing];
              dm += base[dbn * kApproxRing];
            }
          if (odd) { u1 = um; d1 = dm; c1++; } else { u0 = um; d0 = dm; c0++; }
        }
      if (g + 1 < n_groups && !early)
        {
          __syncthreads();
          prefetch (g + 1);
        }
      asm volatile ("cp.async.wait_all;" ::: "memory");
      __syncthreads();                                                      // next group's frames are in; nobody reads this group's any more
    }
  if (s >= n_starts)
    return;
#pragma unroll
  for (int k = 0; k < 2; k++)
    {
      const int bit = 2 * part + k;
      if (bit < n_bits)
        {
          const size_t o = ((size_t) shift_idx * n_starts + s) * n_bits + bit;
          out_ud[o * 2] = k ? u1 : u0;
          out_ud[o * 2 + 1] = k ? d1 : d0;
          out_cnt[o] = k ? c1 : c0;
        }
    }
}

// sync_decode epilogue (bit_quality, src/syncfinder.cc:94-114; normalisation :80-91) + local mean of
// SyncFinder::search_approx (:234-254).  q[i] with i = s*4 + shift is the score list sorted by index.
__global__ void
k_sync_quality (const float *__restrict__ ud, const int *__restrict__ cnt, int n_starts, int n_bits, double norm_div, double *__restrict__ q)
{
  const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 4LL * n_starts)
    return;
  const int s = int (i >> 2), shift_idx = int (i & 3);
  double sync_quality = 0;
  int bit_count = 0;
  for (int bit = 0; bit < n_bits; bit++)
    {
      const size_t o = ((size_t) shift_idx * n_starts + s) * n_bits + bit;
      const float umag = ud[o * 2], dmag = ud[o * 2 + 1];
      double raw_bit;
      if (umag == 0 || dmag == 0)
        raw_bit = 0;
      else if (umag < dmag)
        raw_bit = __fsub_rn (1.0f, __fdiv_rn (umag, dmag));      // float arithmetic as in src/syncfinder.cc:107
      else
        raw_bit = __fsub_rn (__fdiv_rn (dmag, umag), 1.0f);
      sync_quality += ((bit & 1) ? raw_bit : -raw_bit) * cnt[o];
      bit_count += cnt[o];
    }
  if (bit_count)
    sync_quality /= bit_count;
  q[i] = sync_quality / norm_div / 2.9;
}

// local mean of SyncFinder::search_approx (src/syncfinder.cc:234-254) + packing of the score list
__global__ void
k_local_mean (const double *__restrict__ q, long long n, awm_search_score *__restrict__ scores)
{
  const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  double avg = 0;
  int cnt = 0;
  for (int j = -20; j <= 20; j++)
    if (j <= -4 || j >= 4)
      {
        const long long idx = i + j;
        if (idx >= 0 && idx < n)
          {
            avg += q[idx];
            cnt++;
          }
      }
  if (cnt > 0)
    avg /= cnt;
  scores[i].index = (unsigned long long) (i >> 2) * kFrame + (unsigned long long) (i & 3) * 256;
  scores[i].raw_quality = q[i];
  scores[i].local_mean = avg;
}

// local maxima of |raw - local_mean| above a floor, appended in arbitrary order (the host sorts the short list);
// q >= q_last && q >= q_next with 0 beyond the ends (src/syncfinder.cc:258-281; its "skip the next score" rule only
// matters for exactly equal neighbours and is applied by the host).
__global__ void
k_peaks (const awm_search_score *__restrict__ scores, long long n, double floor_q, awm_search_score *__restrict__ out,
         unsigned long long max_out, unsigned long long *__restrict__ counter)
{
  const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  const double q = fabs (scores[i].raw_quality - scores[i].local_mean);
  if (!(q > floor_q))
    return;
  const double q_last = i > 0 ? fabs (scores[i - 1].raw_quality - scores[i - 1].local_mean) : 0;
  const double q_next = i + 1 < n ? fabs (scores[i + 1].raw_quality - scores[i + 1].local_mean) : 0;
  if (q >= q_last && q >= q_next)
    {
      const unsigned long long pos = atomicAdd (counter, 1ull);
      if (pos < max_out)
        out[pos] = scores[i];
    }
}

// =============================================================================================
// SyncFinder::search_refine (src/syncfinder.cc:393-458): for candidate c and fine offset o
// (sample cand_start[c] + 8*o) sync_fft of the wanted sync frames + sync_decode (start frame 0).
// One warp = one (candidate, offset, sync bit): it walks the bit's sync frames in ascending frame order,
// one FFT each, and accumulates umag / dmag in the reference's order (lane 0: up bands, lane 1: down
// bands, sequential float adds), so no spectra are ever written to memory.
// out_ud[((c*65 + o)*n_bits + bit)*2 + {0,1}] = umag, dmag; out_cnt = frames used; out_valid[c*65 + o].
// =============================================================================================
constexpr int kOffsets = 65;
constexpr int kRefineWarps = 10;      // 2 CTAs/SM = 20 warps: shared memory (transpose buffers) and 102 registers/thread both fit

__global__ void __launch_bounds__ (kRefineWarps * 32, 2)
k_refine (const float *__restrict__ pcm, long long n_frames, int C,
          const long long *__restrict__ cand_start, const int *__restrict__ cand_noff, int n_cand,
          const awm_sync_entry *__restrict__ g_ent, const int *__restrict__ g_bit_off, int n_bits, int total_frame_count,
          long long wav_first, long long wav_last,
          float *__restrict__ out_ud, int *__restrict__ out_cnt, unsigned char *__restrict__ out_valid,
          const float2 *g_tw, const float *g_win)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, g_tw, g_win, kRefineWarps);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float *sband = s.extra + w * 96;                      // [81] per warp
  const long long job = (long long) blockIdx.x * kRefineWarps + w;
  if (job >= (long long) n_cand * kOffsets * n_bits)
    return;
  const int c = int (job / (kOffsets * n_bits));
  const int o = int ((job / n_bits) % kOffsets);
  const int bit = int (job % n_bits);
  const long long fine = cand_start[c] + 8LL * o;
  // sync_fft: an offset whose window would read past the end yields no result at all
  const bool valid = o < cand_noff[c] && fine + (long long) total_frame_count * kFrame <= n_frames;
  if (bit == 0 && lane == 0)
    out_valid[c * kOffsets + o] = valid ? 1 : 0;
  if (!valid)
    return;
  float mag = 0.f;                                      // lane 0: umag, lane 1: dmag
  int cnt = 0;
  const int e1 = g_bit_off[bit + 1];
  for (int e = g_bit_off[bit]; e < e1; e++)
    {
      const awm_sync_entry *en = g_ent + e;
      const long long start = fine + (long long) en->frame * kFrame;
      const long long f_first = start * C, f_last = (start + kFrame) * C;
      if (f_last < wav_first || f_first > wav_last)     // frame in digital silence: not counted
        continue;
      float acc[4];
      frame_db_sum (pcm, n_frames, C, start, s, lane, acc);
      bands_to_array (acc, lane, sband, 1);
      __syncwarp();
      if (lane < 2)
        {
          const uint8_t *idx = lane == 0 ? en->up : en->down;
#pragma unroll 6
          for (int i = 0; i < kUD; i++)
            mag += sband[idx[i]];
        }
      cnt++;
      __syncwarp();
    }
  const size_t ob = ((size_t) c * kOffsets + o) * n_bits + bit;
  if (lane < 2)
    out_ud[ob * 2 + lane] = mag;
  if (lane == 0)
    out_cnt[ob] = cnt;
}

// =============================================================================================
// block decode, stage 1: FFTAnalyzer::fft_range (src/wmcommon.cc:123-141) reduced to what
// mix_decode reads: per (block, frame, channel) the dB of bins 20..100 -> D[blk][frame*C+ch][81].
// =============================================================================================
constexpr int kDecodeWarps = 10;

__global__ void __launch_bounds__ (kDecodeWarps * 32, 2)
k_decode_fft (const float *__restrict__ pcm, long long n_frames, int C, const long long *__restrict__ blk_start,
              int n_blk, int frames_per_block, float *__restrict__ D, const float2 *g_tw, const float *g_win)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, g_tw, g_win, kDecodeWarps);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int pairs = (C + 1) / 2;
  const long long job = (long long) blockIdx.x * kDecodeWarps + w;
  const long long per_blk = (long long) frames_per_block * pairs;
  if (job >= per_blk * n_blk)
    return;
  const int b = int (job / per_blk);
  const int f = int ((job % per_blk) / pairs);
  const int chA = int (job % pairs) * 2, chB = chA + 1 < C ? chA + 1 : -1;
  const long long start = blk_start[b] + (long long) f * kFrame;
  float re[32], im[32];
  load_pair (pcm, n_frames, C, start, chA, chB, s.win, re, im, lane);
  const unsigned zero = pair_zero_mask (re, im);
  fft1024_warp (re, im, s.tw, s.xbuf, lane);
  float *da = D + (((size_t) b * frames_per_block + f) * C + chA) * kBands;
  float *dbb = da + kBands;
  float ar, ai, br, bi;
#define AWM_DB(K2) \
  unpack_pair<K2> (re, im, lane, ar, ai, br, bi, zero); \
  { const int band = lane + 32 * K2 - kMinBand; \
    if (band >= 0 && band < kBands) { da[band] = db_from_complex (ar, ai, -96.f); if (chB >= 0) dbb[band] = db_from_complex (br, bi, -96.f); } }
  AWM_DB (0) AWM_DB (1) AWM_DB (2) AWM_DB (3)
#undef AWM_DB
}

// stage 2: mix_decode (src/wmget.cc:67-108) + randomize_bit_order (decode, src/wmcommon.hh:165-185).
// One thread = one coded bit; double accumulators, entries in reference order.
__global__ void
k_mix_decode (const float *__restrict__ D, int n_blk, int C, int frames_per_block,
              const awm_mix_entry *__restrict__ mix, int frames_per_bit, int n_coded,
              const uint16_t *__restrict__ bit_order, float *__restrict__ raw_out)
{
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (o >= n_coded)
    return;
  const float *Db = D + (size_t) b * frames_per_block * C * kBands;
  const long long n_spect = (long long) frames_per_block * C;
  double umag = 0, dmag = 0;
  for (int f = o * frames_per_bit; f < (o + 1) * frames_per_bit; f++)
    for (int ch = 0; ch < C; ch++)
      for (int fb = 0; fb < kUD; fb++)
        {
          const awm_mix_entry me = mix[f * kUD + fb];
          const long long index = (long long) me.frame * C + ch;
          const long long next_index = (index + C) < n_spect ? index + C : index - C;
          const long long prev_index = (index - C) >= 0 ? index - C : index + C;
          const int u = me.up - kMinBand, d = me.down - kMinBand;
          umag += Db[index * kBands + u];
          umag -= double (__fadd_rn (Db[prev_index * kBands + u], Db[next_index * kBands + u])) * 0.5;
          dmag += Db[index * kBands + d];
          dmag -= double (__fadd_rn (Db[prev_index * kBands + d], Db[next_index * kBands + d])) * 0.5;
        }
  raw_out[(size_t) b * n_coded + bit_order[o]] = float (umag - dmag);
}

// =============================================================================================
// normalize_soft_bits (src/wmget.cc:40-65) + conv_decode_soft (src/convcode.cc:128-213).
// One CTA = one code word; decision word u (32 consecutive new states 32u..32u+31) is computed by one thread.
//   new_state ns has predecessors ps0 = ns>>1 and ps1 = ps0 + 2^14; the reference visits old
//   states in ascending order and replaces only on strict '<', so ps1 wins only if strictly better.
//   path metric: delta = (((old + m_0) + m_1) + ...) in float, m_p = (c_p - s_p)^2 as the reference.
// =============================================================================================
constexpr int kVitStates = 1 << AWM_VITERBI_ORDER;
constexpr int kVitThreads = 512;      // CTA size; each thread owns two groups of 32 new states
constexpr int kVitWords = kVitStates / 32;   // decision words per trellis step

// generator polynomials (src/convcode.cc:42-46) as compile-time constants: A = even, B = odd, AB = all
__host__ __device__ constexpr unsigned ab_generator (int i)
{
  return i == 0 ? 066561u : i == 1 ? 075211u : i == 2 ? 071545u : i == 3 ? 054435u : i == 4 ? 063635u : i == 5 ? 052475u
       : i == 6 ? 063543u : i == 7 ? 075307u : i == 8 ? 052547u : i == 9 ? 045627u : i == 10 ? 067657u : 051757u;
}
template<int TYPE> __host__ __device__ constexpr unsigned type_generator (int p) { return TYPE == AWM_BLOCK_AB ? ab_generator (p) : ab_generator (2 * p + TYPE); }
__host__ __device__ constexpr bool cparity (unsigned v) { v ^= v >> 16; v ^= v >> 8; v ^= v >> 4; v ^= v >> 2; v ^= v >> 1; return v & 1u; }

// One trellis step for the 32 new states ns = 32u + q of group u; returns the 32 decision bits.
// The output bit p of state ns is parity (ns & g_p) = parity (32u & g_p) ^ parity (q & g_p): the first factor
// is a per-group constant (hi, bit p), the second a compile-time constant, so which of (c-0)^2 / (c-1)^2 is
// added needs no instruction at all inside the unrolled loops.
// shared-memory position of path metric n: four floats of padding after every 32, so that the float4 accesses of a quarter warp
// (reads 64 bytes apart, writes 128 bytes apart in the unpadded array) fall into eight different bank groups
__device__ __forceinline__ int vit_pos (int n) { return n + ((n >> 5) << 2); }
constexpr int kVitPadded = kVitStates + kVitStates / 32 * 4;

// d_lo / d_hi: the path metrics of the predecessors ps0 = 16 u + .. (lower half of the states) and ps1 = ps0 + 2^14 (upper half),
// both addressed with vit_pos (16 u + ..)
template<int TYPE> __device__ __forceinline__ uint32_t
viterbi_step (const float *__restrict__ d_lo, const float *__restrict__ d_hi, float (&outv)[32], unsigned hi, const float *m0, const float *m1, int u)
{
  constexpr int RATE = TYPE == AWM_BLOCK_AB ? 12 : 6;
  // The two candidates of a new state -- coming from predecessor ps0 and from ps1 -- add the SAME branch metrics in the same order,
  // so they travel as one packed pair (d0, d1) and every step of the sum is one FADD2 (add.rn.f32x2: both halves rounded exactly like
  // __fadd_rn) instead of two FADDs: the add-compare-select loop issues half the instructions, bit-identical metrics.
  f2 mA[RATE], mB[RATE];                  // (m, m): metric for output bit == hi-bit / != hi-bit
#pragma unroll
  for (int p = 0; p < RATE; p++)
    {
      const bool h = (hi >> p) & 1u;
      const float a = h ? m1[p] : m0[p], b = h ? m0[p] : m1[p];
      mA[p] = f2_make (a, a);
      mB[p] = f2_make (b, b);
    }
  uint32_t word = 0;
#pragma unroll
  for (int v = 0; v < 4; v++)                                // 8 new states <- 4 + 4 predecessors
    {
      const float4 x = *reinterpret_cast<const float4 *> (d_lo + vit_pos (16 * u + 4 * v));
      const float4 y = *reinterpret_cast<const float4 *> (d_hi + vit_pos (16 * u + 4 * v));
      const f2 a01[4] = { f2_make (x.x, y.x), f2_make (x.y, y.y), f2_make (x.z, y.z), f2_make (x.w, y.w) };
#pragma unroll
      for (int q = 0; q < 8; q++)
        {
          f2 d = a01[q >> 1];
#pragma unroll
          for (int p = 0; p < RATE; p++)
            d = f2_add (d, cparity (unsigned (8 * v + q) & type_generator<TYPE> (p)) ? mB[p] : mA[p]);
          float d0, d1;
          f2_split (d, d0, d1);
          const bool take1 = d1 < d0;
          outv[8 * v + q] = take1 ? d1 : d0;
          word |= (take1 ? 1u : 0u) << (8 * v + q);
        }
    }
  return word;
}

// The 2^15 path metrics of a code word live in shared memory (128 KB).  A trellis step reads the two predecessors of every new
// state, so the update cannot be done in place state by state; instead every thread keeps the 64 new metrics of its two groups in
// registers until the whole CTA has read the old ones (barrier), then stores them over the old array (barrier).  No metric ever
// travels to L2 / HBM; only the decision bits (4 KB per step, read back once by the traceback) are written to global memory.
template<int TYPE> __device__ __forceinline__ void
viterbi_run (float *dm, uint32_t *dec, const float *coded, float *m0, float *m1, int steps, int tid)
{
  constexpr int RATE = TYPE == AWM_BLOCK_AB ? 12 : 6;
  constexpr int kGroups = kVitWords / kVitThreads;
  unsigned hi[kGroups];
#pragma unroll
  for (int g = 0; g < kGroups; g++)
    {
      const unsigned base = 32u * unsigned (tid + g * kVitThreads);
      hi[g] = 0;
#pragma unroll
      for (int p = 0; p < RATE; p++)
        hi[g] |= unsigned (__popc (base & type_generator<TYPE> (p)) & 1) << p;
    }
  for (int t = 0; t < steps; t++)
    {
      if (tid < RATE)
        {
          const float c = coded[t * RATE + tid];
          m0[tid] = __fmul_rn (c, c);                       // (c - 0)^2
          m1[tid] = __fmul_rn (c - 1.0f, c - 1.0f);         // (c - 1)^2
        }
      __syncthreads();                                      // metrics of the previous step stored, m0 / m1 ready
      float outv[kGroups][32];
#pragma unroll
      for (int g = 0; g < kGroups; g++)
        {
          const int u = tid + g * kVitThreads;
          dec[(size_t) t * kVitWords + u] = viterbi_step<TYPE> (dm, dm + vit_pos (kVitStates >> 1), outv[g], hi[g], m0, m1, u);
        }
      __syncthreads();                                      // every thread has read its predecessors
#pragma unroll
      for (int g = 0; g < kGroups; g++)
        {
          float4 *on = reinterpret_cast<float4 *> (dm + vit_pos (32 * (tid + g * kVitThreads)));
#pragma unroll
          for (int k = 0; k < 8; k++)
            on[k] = make_float4 (outv[g][4 * k], outv[g][4 * k + 1], outv[g][4 * k + 2], outv[g][4 * k + 3]);
        }
    }
  __syncthreads();
}

/* Traceback (src/convcode.cc:192-211) by one warp.  Going back one step reads ONE decision bit, but which word of the previous step
 * holds it depends on the bit just read: done by one thread this is a chain of 143 dependent global loads.  The word index of step
 * t - 1 - k is (state >> (5 + k)) | (the k decisions in between) << (10 - k): the warp loads the word of step t - 1 and all
 * 2 + 4 + 8 + 16 candidate words of the four steps before it at once (31 lanes, one load latency), then walks the five steps through
 * shuffles. */
__device__ __forceinline__ void
viterbi_traceback (const uint32_t *dec, int steps, int n_msg, unsigned char *bits_out, int lane)
{
  unsigned state = 0;
  int t = steps;
  while (t > 0)
    {
      const int depth = t < 5 ? t : 5;                  // steps resolved in this round
      /* lane 2^k - 1 + c (k = 0 .. 4, c < 2^k): candidate c of step t - 1 - k, c = the k decisions read so far, newest in the lowest bit */
      int k = 31 - __clz (lane + 1);
      const unsigned c = unsigned (lane + 1) - (1u << k);
      uint32_t word = 0;
      if (lane < 31 && k < depth)
        {
          unsigned rev = 0;                               // decisions enter the state from the top: oldest decision lowest
          for (int i = 0; i < k; i++)
            rev |= ((c >> i) & 1u) << (k - 1 - i);
          const unsigned widx = ((state >> (5 + k)) | (rev << (10 - k))) & (kVitWords - 1);
          word = dec[(size_t) (t - 1 - k) * kVitWords + widx];
        }
      unsigned path = 0;                                  // decisions of this round, newest in the lowest bit
      for (k = 0; k < depth; k++)
        {
          const uint32_t w = __shfl_sync (0xffffffffu, word, (1 << k) - 1 + int (path));
          const unsigned sel = (w >> (state & 31)) & 1u;
          if (lane == 0 && t - 1 - k < n_msg)
            bits_out[t - 1 - k] = state & 1u;
          state = (state >> 1) | (sel << (AWM_VITERBI_ORDER - 1));
          path = (path << 1) | sel;
        }
      t -= depth;
    }
}

constexpr size_t viterbi_smem_bytes (int steps) { return size_t (kVitPadded) * sizeof (float) + size_t (steps) * 12 * sizeof (float); }

__global__ void __launch_bounds__ (kVitThreads)
k_viterbi (const float *__restrict__ raw, const long long *__restrict__ raw_off, int n_msg, const int *__restrict__ block_types, int hard,
           int max_steps, uint32_t *__restrict__ dec_buf /* [job][steps][kVitWords] */,
           unsigned char *__restrict__ bits_out, float *__restrict__ err_out)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  float *dm = reinterpret_cast<float *> (smem);             // [2^15] path metrics (padded, vit_pos)
  float *coded = dm + kVitPadded;                           // [n_coded] normalised soft bits
  __shared__ float m0[12], m1[12];
  __shared__ double s_mean;
  const int job = blockIdx.x, tid = threadIdx.x;
  const int btype = block_types[job];
  const int rate = (btype == AWM_BLOCK_AB) ? 12 : 6;
  const int steps = n_msg + AWM_VITERBI_ORDER;
  const int n_coded = steps * rate;

  const float *rj = raw + raw_off[job];
  if (tid == 0)
    {
      double mean = 0;
      for (int i = 0; i < n_coded; i++)
        mean += fabs (double (rj[i]));
      s_mean = mean / n_coded;
    }
  __syncthreads();
  /* digital silence: every raw soft bit is exactly 0, so mean == 0 and normalize_soft_bits (src/wmget.cc:56-61) yields 0/0 = NaN for
   * every coded bit (raw values are finite sums of dB values, so NaN is all-or-nothing).  In conv_decode_soft (src/convcode.cc:164-190)
   * the NaN path metrics of step 0 fail the "old_table[state].delta >= 0" reachability test of step 1: every later table keeps its
   * initial StateEntry {0, -1, 0}, the traceback reads bit 0 / last_state 0 everywhere and error_out = -1 / n_coded. */
  if (!hard && !(s_mean > 0))
    {
      for (int i = tid; i < n_msg; i += blockDim.x)
        bits_out[(size_t) job * n_msg + i] = 0;
      if (tid == 0)
        err_out[job] = -1.0f / float (n_coded);
      return;
    }
  for (int i = tid; i < n_coded; i += blockDim.x)
    coded[i] = hard ? (rj[i] > 0 ? 1.0f : 0.0f) : float (0.5 * (double (rj[i]) / s_mean + 1));

  uint32_t *dec = dec_buf + (size_t) job * max_steps * kVitWords;
  for (int i = tid; i < kVitStates; i += blockDim.x)
    dm[vit_pos (i)] = (i == 0) ? 0.f : INFINITY;
  __syncthreads();

  if (btype == AWM_BLOCK_A)
    viterbi_run<AWM_BLOCK_A> (dm, dec, coded, m0, m1, steps, tid);
  else if (btype == AWM_BLOCK_B)
    viterbi_run<AWM_BLOCK_B> (dm, dec, coded, m0, m1, steps, tid);
  else
    viterbi_run<AWM_BLOCK_AB> (dm, dec, coded, m0, m1, steps, tid);
  if (tid == 0)
    err_out[job] = dm[0] / float (n_coded);
  if (tid < 32)
    viterbi_traceback (dec, steps, n_msg, bits_out + (size_t) job * n_msg, tid);
}

// =============================================================================================
// embed: FFTAnalyzer::run_fft (src/wmcommon.cc:91-121) + apply_frame_mod (src/wmadd.cc:61-84) +
// WatermarkSynth::run (src/wmadd.cc:215-250) + "samples[i] += orig_samples[i]" (src/wmadd.cc:564-565)
// + Limiter::block_max (src/limiter.cc:90-97), fused.  CTA = 16 warps = 14 output frames + one halo
// frame on each side (output frame m needs the synthesis-window tails of frames m-1 and m+1,
// ~103 samples each, which travel through shared memory).
// =============================================================================================
constexpr int kEmbedWarps = 16;
constexpr int kEmbedTile = kEmbedWarps - 2;
constexpr int kEdge = 104;            // synthesis window is non-zero for x < 103 (tail) and x > 921 (head)
constexpr int kEdgeHi = kFrame - kEdge;

struct EmbedArgs
{
  const float *in;
  float *out;
  long long n_frames;          // valid input sample-frames
  int C;
  long long n_proc;            // 1024-frames to process = ceil(n/1024) + 1 (tail spill)
  long long frame_begin, frame_end;   // this launch emits frames [frame_begin, frame_end) (pipelined host<->device copies launch pieces)
  long long frame_number0;     // table row counter of frame 0: first_frame_number + 2*fpb - pad_start
  int fpb;
  const uint8_t *frame_mod;    // [2][fpb][101]
  float pow_up, pow_down;      // HALF the exponents -delta*(+1), -delta*(-1): applied to log2 of the squared magnitude
  int limiter_block;           // 0 = no peak tracking
  long long stream_pos0;       // stream position of sample 0 of this buffer (first_frame_number * 1024): limiter blocks are stream-global
  long long blk0;              // stream_pos0 / limiter_block: peaks[] is indexed relative to it
  unsigned *peaks;             // [n_blocks] float bits, atomicMax
  double *snr;                 // [2] or null
  long long snr_frames;        // frames that count for --snr (the reference loop stops earlier without limiter)
  long long snr_pos0, snr_pos1; // ... and only positions [snr_pos0, snr_pos1) of this buffer (a window of a longer stream counts its own part)
  int delta_only;              // 1: write the watermark signal alone (WatermarkGen::run output), not input + watermark
  const float2 *tw;
  const float *win;
  const float *synth;          // [3072] synthesis window
};

// delta spectrum of one K2 group (bins lane + 32 K2 of both channels of the pair) written into the (re <-> im swapped) input of the
// inverse transform, mirrored half included.  Shared by k_embed and k_embed_strip; every product and sum is spelled out with its
// rounding (no FMA contraction left to the compiler), so the two kernels produce identical bits.
template<int K2> __device__ __forceinline__ void
embed_mod_group (const float (&re)[32], const float (&im)[32], float (&inr)[32], float (&ini)[32], const uint8_t *fm,
                 float pow_up, float pow_down, bool have_b, int lane)
{
  float ar, ai, br, bi;
  unpack_pair<K2> (re, im, lane, ar, ai, br, bi);
  const int k = lane + 32 * K2;
  float dar = 0.f, dai = 0.f, dbr = 0.f, dbi = 0.f;
  if (k >= kMinBand && k <= kMaxBand)
    {
      const int mod = fm[k];
      if (mod != 0)
        {
          /* mag^e - 1 = exp2 (e/2 * log2 (re^2 + im^2)) - 1; mag > 1e-7 <=> mag^2 > 1e-14 */
          const float ex2 = (mod == 1) ? pow_up : pow_down;
          const float pa = __fmaf_rn (ar, ar, __fmul_rn (ai, ai));
          if (pa > 1e-14f)
            {
              const float f = __fsub_rn (exp2f (__fmul_rn (ex2, log2f (pa))), 1.0f);
              dar = __fmul_rn (ar, f);
              dai = __fmul_rn (ai, f);
            }
          if (have_b)
            {
              const float pb = __fmaf_rn (br, br, __fmul_rn (bi, bi));
              if (pb > 1e-14f)
                {
                  const float f = __fsub_rn (exp2f (__fmul_rn (ex2, log2f (pb))), 1.0f);
                  dbr = __fmul_rn (br, f);
                  dbi = __fmul_rn (bi, f);
                }
            }
        }
    }
  /* D[k] = dA + i dB ; D[N-k] = conj dA + i conj dB ; registers hold the re<->im swapped input */
  inr[K2] = __fadd_rn (dai, dbr);
  ini[K2] = __fsub_rn (dar, dbi);
  const float mr = __fadd_rn (dar, dbi), mi = __fsub_rn (dbr, dai);
  const int src = (32 - lane) & 31;
  const float gr = __shfl_sync (0xffffffffu, mr, src), gi = __shfl_sync (0xffffffffu, mi, src);
  if (lane == 0) { inr[(32 - K2) & 31] = (K2 == 0) ? inr[0] : gi; ini[(32 - K2) & 31] = (K2 == 0) ? ini[0] : gr; }
  else           { inr[31 - K2] = gi; ini[31 - K2] = gr; }
}

__global__ void __launch_bounds__ (kEmbedWarps * 32, 1)
k_embed (EmbedArgs A)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, A.tw, A.win, kEmbedWarps);
  float *synth = s.extra;                                   // [3072]
  float2 *elo = reinterpret_cast<float2 *> (synth + 3 * kFrame);  // [warps][kEdge]   samples x < kEdge
  float2 *ehi = elo + kEmbedWarps * kEdge;                  // [warps][kEdge]   samples x >= kEdgeHi
  for (int i = threadIdx.x; i < 3 * kFrame; i += blockDim.x)
    synth[i] = A.synth[i];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long m = A.frame_begin + (long long) blockIdx.x * kEmbedTile - 1 + w;      // frame handled by this warp
  const long long n_real = (A.n_frames + kFrame - 1) / kFrame;          // frames that contain input
  const bool exists = m >= 0 && m < n_real;
  const bool emits = w >= 1 && w <= kEmbedTile && m >= A.frame_begin && m < A.frame_end && m < A.n_proc;
  const int C = A.C;
  float pk0 = 0.f, pk1 = 0.f;
  double snr_d = 0, snr_s = 0;
  long long blk_lo = 0, boundary = 0;
  if (A.limiter_block > 0 && emits)
    {
      const long long gpos = A.stream_pos0 + m * kFrame;
      blk_lo = gpos / A.limiter_block;
      boundary = (blk_lo + 1) * A.limiter_block - gpos;                // x >= boundary belongs to the next block
      blk_lo -= A.blk0;
    }

  for (int chA = 0; chA < C; chA += 2)
    {
      const int chB = chA + 1 < C ? chA + 1 : -1;
      float re[32], im[32];
      __syncthreads();                                      // synth[] ready / previous pair's edges consumed
      if (exists)
        {
          load_pair (A.in, A.n_frames, C, m * kFrame, chA, chB, s.win, re, im, lane);
          fft1024_warp (re, im, s.tw, s.xbuf, lane);
          const long long r = (A.frame_number0 + m) % (2LL * A.fpb);
          const uint8_t *fm = A.frame_mod + (size_t) r * (kMaxBand + 1);   // rows [0,fpb) = A, [fpb,2fpb) = B
          float inr[32], ini[32];
#pragma unroll
          for (int j = 0; j < 32; j++)
            inr[j] = ini[j] = 0.f;
          // own bins k = lane + 32*K2 at register K2, mirrored bins N-k arrive from lane (32-lane)&31
          embed_mod_group<0> (re, im, inr, ini, fm, A.pow_up, A.pow_down, chB >= 0, lane);
          embed_mod_group<1> (re, im, inr, ini, fm, A.pow_up, A.pow_down, chB >= 0, lane);
          embed_mod_group<2> (re, im, inr, ini, fm, A.pow_up, A.pow_down, chB >= 0, lane);
          embed_mod_group<3> (re, im, inr, ini, fm, A.pow_up, A.pow_down, chB >= 0, lane);
          fft1024_warp (inr, ini, s.tw, s.xbuf, lane);
          // inverse result: sample x = lane + 32*brev5(i): channel A = ini[i], channel B = inr[i]
#pragma unroll
          for (int i = 0; i < 32; i++)
            {
              re[i] = ini[i];
              im[i] = inr[i];
            }
        }
      else
        {
#pragma unroll
          for (int i = 0; i < 32; i++)
            re[i] = im[i] = 0.f;
        }
      // publish the window tails
#pragma unroll
      for (int i = 0; i < 32; i++)
        {
          const int x = lane + 32 * brev5 (i);
          if (x < kEdge)
            elo[w * kEdge + x] = make_float2 (re[i], im[i]);
          if (x >= kEdgeHi)
            ehi[w * kEdge + (x - kEdgeHi)] = make_float2 (re[i], im[i]);
        }
      __syncthreads();
      if (emits)
        {
#pragma unroll
          for (int i = 0; i < 32; i++)
            {
              const int x = lane + 32 * brev5 (i);
              // wm = ((0 + prev*w2) + cur*w1) + next*w0, every product and sum rounded separately (src/wmadd.cc:228-238)
              float wa = __fmul_rn (re[i], synth[kFrame + x]);
              float wb = __fmul_rn (im[i], synth[kFrame + x]);
              if (x < kEdge)
                {
                  const float2 p = elo[(w - 1) * kEdge + x];
                  wa = __fadd_rn (__fmul_rn (p.x, synth[2 * kFrame + x]), wa);
                  wb = __fadd_rn (__fmul_rn (p.y, synth[2 * kFrame + x]), wb);
                }
              if (x >= kEdgeHi)
                {
                  const float2 nx = ehi[(w + 1) * kEdge + (x - kEdgeHi)];
                  wa = __fadd_rn (wa, __fmul_rn (nx.x, synth[x]));
                  wb = __fadd_rn (wb, __fmul_rn (nx.y, synth[x]));
                }
              const long long pos = m * kFrame + x;
              float oa = 0.f, ob = 0.f;
              if (pos < A.n_frames)
                {
                  if (C == 2)
                    {
                      const float2 v = __ldg (reinterpret_cast<const float2 *> (A.in) + pos);
                      oa = v.x; ob = v.y;
                    }
                  else
                    {
                      oa = __ldg (A.in + pos * C + chA);
                      if (chB >= 0)
                        ob = __ldg (A.in + pos * C + chB);
                    }
                }
              const float ya = A.delta_only ? wa : __fadd_rn (wa, oa), yb = A.delta_only ? wb : __fadd_rn (wb, ob);
              if (A.snr && m < A.snr_frames && pos >= A.snr_pos0 && pos < A.snr_pos1)
                {
                  snr_d += double (wa) * double (wa) + (chB >= 0 ? double (wb) * double (wb) : 0.0);
                  snr_s += double (oa) * double (oa) + (chB >= 0 ? double (ob) * double (ob) : 0.0);
                }
              float mx = fabsf (ya);
              if (chB >= 0)
                mx = fmaxf (mx, fabsf (yb));
              if (x < boundary) pk0 = fmaxf (pk0, mx); else pk1 = fmaxf (pk1, mx);
              if (pos < A.n_frames)
                {
                  if (C == 2)
                    reinterpret_cast<float2 *> (A.out)[pos] = make_float2 (ya, yb);
                  else
                    {
                      A.out[pos * C + chA] = ya;
                      if (chB >= 0)
                        A.out[pos * C + chB] = yb;
                    }
                }
            }
        }
    }
  if (A.limiter_block > 0 && emits)
    {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1)
        {
          pk0 = fmaxf (pk0, __shfl_xor_sync (0xffffffffu, pk0, off));
          pk1 = fmaxf (pk1, __shfl_xor_sync (0xffffffffu, pk1, off));
        }
      if (lane == 0)
        {
          atomicMax (A.peaks + blk_lo, __float_as_uint (pk0));
          if (boundary < kFrame)
            atomicMax (A.peaks + blk_lo + 1, __float_as_uint (pk1));
        }
    }
  if (A.snr && emits)
    {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1)
        {
          snr_d += __shfl_xor_sync (0xffffffffu, snr_d, off);
          snr_s += __shfl_xor_sync (0xffffffffu, snr_s, off);
        }
      if (lane == 0)
        {
          atomicAdd (A.snr, snr_d);
          atomicAdd (A.snr + 1, snr_s);
        }
    }
}

// Limiter::process_block (src/limiter.cc:99-124): gain ramps linearly over each block between
// ceiling / max (bm[b-1], bm[b]) and ceiling / max (bm[b], bm[b+1]); bm[b] = max (ceiling, peak[b]).
constexpr int kLimiterIter = 16;        // sample-frames per thread: a CTA covers 4096 consecutive positions

__global__ void
k_limiter (float *__restrict__ x, long long pos_begin, long long pos_end, int C, int block, float ceiling,
           const unsigned *__restrict__ peaks, long long n_blocks, long long stream_pos0)
{
  const long long cta_first = pos_begin + (long long) blockIdx.x * blockDim.x * kLimiterIter;
  if (cta_first >= pos_end)
    return;
  // most audio never reaches the ceiling: if no limiter block that touches this CTA's range (or its neighbours, which steer the
  // gain ramp) has a peak above it, every scale factor is exactly 1.0 and x * 1.0f == x -- nothing to read or write
  {
    const long long cta_last = (cta_first + (long long) blockDim.x * kLimiterIter < pos_end ? cta_first + (long long) blockDim.x * kLimiterIter : pos_end) - 1;
    const long long b_lo = (stream_pos0 + cta_first) / block - stream_pos0 / block - 1, b_hi = (stream_pos0 + cta_last) / block - stream_pos0 / block + 1;
    bool engaged = false;
    for (long long b = b_lo < 0 ? 0 : b_lo; b <= b_hi && b < n_blocks; b++)
      if (__uint_as_float (peaks[b]) > ceiling)
        engaged = true;
    if (!engaged)
      return;
  }
  for (int it = 0; it < kLimiterIter; it++)
    {
      const long long pos = cta_first + (long long) it * blockDim.x + threadIdx.x;
      if (pos >= pos_end)
        return;
      const long long gpos = stream_pos0 + pos;
      const long long b = gpos / block - stream_pos0 / block;           // index into peaks[]
      const int i = int (gpos % block);
      const float cur = fmaxf (ceiling, __uint_as_float (peaks[b]));
      // block -1 of the stream counts as "ceiling"; for a shard that starts mid-stream the caller's halo makes peaks[b-1] valid
      const float last = b > 0 ? fmaxf (ceiling, __uint_as_float (peaks[b - 1])) : ceiling;
      const float next = b + 1 < n_blocks ? fmaxf (ceiling, __uint_as_float (peaks[b + 1])) : ceiling;
      const float scale_start = __fdiv_rn (ceiling, fmaxf (last, cur));
      const float scale_end = __fdiv_rn (ceiling, fmaxf (cur, next));
      if (scale_start == 1.0f && scale_end == 1.0f)
        continue;                                               // x * 1.0f == x
      const float scale_step = __fdiv_rn (__fsub_rn (scale_end, scale_start), float (block));
      const float scale = __fadd_rn (scale_start, __fmul_rn (float (i), scale_step));
      for (int c = 0; c < C; c++)
        x[pos * C + c] = __fmul_rn (x[pos * C + c], scale);
    }
}

} // namespace awm
