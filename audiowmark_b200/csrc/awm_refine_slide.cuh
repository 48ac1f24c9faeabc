// awm_refine_slide.cuh -- SyncFinder::search_refine (src/syncfinder.cc:393-458) with a sliding DFT.
//
// search_refine scores 65 fine offsets (8 samples apart) per candidate; for each of them the reference transforms all
// wanted sync frames again (sync_fft, :560-605) although consecutive offsets share 1016 of the 1024 samples of every frame.
// Here one warp owns one (candidate, sync frame) pair and walks the 65 offsets:
//   offset 0     : one 1024-point FFT of the un-windowed frame (left + i right) -> rectangular-window spectrum R[k], k = 19..102
//   offset m+1   : R'[k] = W^(-8k) (R[k] + sum_{j<8} (x[P+1024+j] - x[P+j]) W^(jk)),  W = exp (-2 pi i / 1024)
//   Hann window  : the reference's window w[n] = (0.5 - 0.5 cos (2 pi n / 1024)) / 256 acts in the frequency domain as
//                  X[k] = (R[k] - (R[k-1] + R[k+1]) / 2) / 512
//   dB of bins 20..100 summed over the channels, up / down band sums of this sync frame (warp reduction)
// ~290 warp instructions per offset instead of ~1700 for a fresh transform.  A second kernel adds the per-frame sums of each
// sync bit in frame order.  Numerics: a float sliding update carries an error of a few 1e-6 relative to the largest
// bins after 64 steps, the same order as a float FFT's own rounding (DESIGN.md section 6); tests hold it to the
// same bars as the FFT path (quality 2e-4, index within one 8-sample step).
// Lane l keeps bins 19 + 3l .. 21 + 3l (lanes 0..27), so the Hann neighbours are one shuffle away.
#pragma once
#include "awm_kernels.cuh"

namespace awm {

constexpr int kSlideWarps = 8;
constexpr int kSlideBins = 3;

template<int C> __global__ void __launch_bounds__ (kSlideWarps * 32, 2)
k_refine_slide (const float *__restrict__ pcm, long long n_frames,
                const long long *__restrict__ cand_start, const int *__restrict__ cand_noff, int n_cand,
                const awm_sync_entry *__restrict__ g_ent, int n_ent, int total_frame_count,
                long long wav_first, long long wav_last,
                float2 *__restrict__ ent_ud /* [cand][65][n_ent] */, unsigned char *__restrict__ ent_flag,
                const float2 *g_tw, const float2 *__restrict__ tw1024)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, g_tw, nullptr, kSlideWarps);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long job = (long long) blockIdx.x * kSlideWarps + w;
  if (job >= (long long) n_cand * n_ent)
    return;
  const int c = int (job / n_ent), e = int (job % n_ent);
  const awm_sync_entry *en = g_ent + e;
  const long long p0 = cand_start[c] + (long long) en->frame * kFrame;      // first sample of this sync frame at offset 0
  // offsets whose block would read past the end yield no result (sync_fft returns nothing): same rule as k_refine
  long long n_valid = cand_noff[c];
  {
    const long long room = n_frames - (long long) total_frame_count * kFrame - cand_start[c];
    n_valid = room < 0 ? 0 : (n_valid < room / 8 + 1 ? n_valid : room / 8 + 1);
  }
  float2 *out = ent_ud + ((size_t) c * kOffsets) * n_ent + e;
  unsigned char *flag = ent_flag + ((size_t) c * kOffsets) * n_ent + e;
  if (n_valid <= 0)
    return;

  // ---- offset 0: rectangular-window spectrum by one FFT
  float rl_re[kSlideBins], rl_im[kSlideBins], rr_re[kSlideBins], rr_im[kSlideBins];
  {
    float re[32], im[32];
    if (C == 2)
      {
        const float2 *p = reinterpret_cast<const float2 *> (pcm) + p0 + lane;
#pragma unroll
        for (int j = 0; j < 32; j++)
          {
            const float2 v = __ldg (p + 32 * j);
            re[j] = v.x;
            im[j] = v.y;
          }
      }
    else
      {
#pragma unroll
        for (int j = 0; j < 32; j++)
          {
            re[j] = __ldg (pcm + p0 + 32 * j + lane);
            im[j] = 0.f;
          }
      }
    const unsigned zero = pair_zero_mask (re, im);      // a channel that is zero over the frame slides on from an exactly zero spectrum
    fft1024_warp (re, im, s.tw, s.xbuf, lane);
    float4 *sc = reinterpret_cast<float4 *> (s.xbuf);           // the transpose buffer is free again: [128] (Lre, Lim, Rre, Rim)
    float ar, ai, br, bi;
    unpack_pair<0> (re, im, lane, ar, ai, br, bi, zero); sc[lane]      = make_float4 (ar, ai, br, bi);
    unpack_pair<1> (re, im, lane, ar, ai, br, bi, zero); sc[lane + 32] = make_float4 (ar, ai, br, bi);
    unpack_pair<2> (re, im, lane, ar, ai, br, bi, zero); sc[lane + 64] = make_float4 (ar, ai, br, bi);
    unpack_pair<3> (re, im, lane, ar, ai, br, bi, zero); sc[lane + 96] = make_float4 (ar, ai, br, bi);
    __syncwarp();
#pragma unroll
    for (int b = 0; b < kSlideBins; b++)
      {
        const int k = (19 + kSlideBins * lane + b) & 127;
        const float4 v = sc[k];
        rl_re[b] = v.x; rl_im[b] = v.y; rr_re[b] = v.z; rr_im[b] = v.w;
      }
    __syncwarp();
  }
  // ---- per-lane constants: W^(jk) for the 8 entering / leaving samples, the rotation W^(-8k), band membership
  float wr[kSlideBins][8], wi[kSlideBins][8], rot_c[kSlideBins], rot_s[kSlideBins], m_up[kSlideBins], m_dn[kSlideBins];
#pragma unroll
  for (int b = 0; b < kSlideBins; b++)
    {
      const int k = 19 + kSlideBins * lane + b;
#pragma unroll
      for (int j = 0; j < 8; j++)
        {
          const float2 t = __ldg (tw1024 + ((j * k) & 1023));
          wr[b][j] = t.x;
          wi[b][j] = t.y;
        }
      const float2 r = __ldg (tw1024 + ((8 * k) & 1023));
      rot_c[b] = r.x;
      rot_s[b] = -r.y;                     // conj: W^(-8k)
      const int band = k - kMinBand;
      float mu = 0.f, md = 0.f;
      if (band >= 0 && band < kBands)
        for (int i = 0; i < kUD; i++)
          {
            if (en->up[i] == band) mu = 1.f;
            if (en->down[i] == band) md = 1.f;
          }
      m_up[b] = mu;
      m_dn[b] = md;
    }

  // The 16 samples that enter / leave the frame at the next slide are loaded one iteration ahead: their latency hides behind the Hann /
  // dB / reduction work of the current offset instead of stalling the first subtraction of the slide (17 % of this kernel's stall
  // samples before).  The address is clamped to the last slide that exists, so the load itself needs no predicate.
  auto load_delta = [&] (long long m, float (&dl)[8], float (&dr)[8])
    {
      const long long mm = m + 1 < n_valid ? m : (n_valid >= 2 ? n_valid - 2 : 0);
      const long long start = p0 + 8 * mm;
      if (C == 2)
        {
          const float2 *po = reinterpret_cast<const float2 *> (pcm) + start;
#pragma unroll
          for (int j = 0; j < 8; j++)
            {
              const float2 xo = __ldg (po + j), xi = __ldg (po + kFrame + j);
              dl[j] = xi.x - xo.x;
              dr[j] = xi.y - xo.y;
            }
        }
      else
        {
#pragma unroll
          for (int j = 0; j < 8; j++)
            {
              dl[j] = __ldg (pcm + start + kFrame + j) - __ldg (pcm + start + j);
              dr[j] = 0.f;
            }
        }
    };
  // dB for RANKING the offsets: MUFU.LG2 (__log2f, abs. error ~1e-7 on these magnitudes -- an order below the float sliding DFT's own
  // error) instead of the ~22-instruction log2f; the offsets that matter are scored again exactly by k_refine_exact_*
  auto db_fast = [] (float abs2) { return abs2 > 0.0f ? __log2f (abs2) * 3.01029995663981f : -96.0f; };
  if (n_valid > 1 && p0 + 8 * (n_valid - 2) + kFrame + 8 > n_frames)       // cannot happen (n_valid is cut to the stream above); keeps the loads in bounds
    return;
  for (long long m = 0; m < n_valid; m++)
    {
      const long long start = p0 + 8 * m;
      float dl[8], dr[8];
      if (n_valid > 1)
        load_delta (m, dl, dr);
      // ---- Hann in the frequency domain + dB + band sums
      const float ll_re = __shfl_up_sync (0xffffffffu, rl_re[2], 1), ll_im = __shfl_up_sync (0xffffffffu, rl_im[2], 1);
      const float nl_re = __shfl_down_sync (0xffffffffu, rl_re[0], 1), nl_im = __shfl_down_sync (0xffffffffu, rl_im[0], 1);
      float lr_re = 0, lr_im = 0, nr_re = 0, nr_im = 0;
      if (C == 2)
        {
          lr_re = __shfl_up_sync (0xffffffffu, rr_re[2], 1); lr_im = __shfl_up_sync (0xffffffffu, rr_im[2], 1);
          nr_re = __shfl_down_sync (0xffffffffu, rr_re[0], 1); nr_im = __shfl_down_sync (0xffffffffu, rr_im[0], 1);
        }
      float u = 0.f, d = 0.f;
#pragma unroll
      for (int b = 0; b < kSlideBins; b++)
        {
          const float pl_re = b == 0 ? ll_re : rl_re[b - 1], pl_im = b == 0 ? ll_im : rl_im[b - 1];
          const float ql_re = b == kSlideBins - 1 ? nl_re : rl_re[b + 1], ql_im = b == kSlideBins - 1 ? nl_im : rl_im[b + 1];
          const float hl_re = rl_re[b] - 0.5f * (pl_re + ql_re), hl_im = rl_im[b] - 0.5f * (pl_im + ql_im);
          // (1/512)^2 on the squared magnitude: exact power of two, same value as scaling the spectrum first
          float db = db_fast ((hl_re * hl_re + hl_im * hl_im) * 3.814697265625e-06f);
          if (C == 2)
            {
              const float pr_re = b == 0 ? lr_re : rr_re[b - 1], pr_im = b == 0 ? lr_im : rr_im[b - 1];
              const float qr_re = b == kSlideBins - 1 ? nr_re : rr_re[b + 1], qr_im = b == kSlideBins - 1 ? nr_im : rr_im[b + 1];
              const float hr_re = rr_re[b] - 0.5f * (pr_re + qr_re), hr_im = rr_im[b] - 0.5f * (pr_im + qr_im);
              db += db_fast ((hr_re * hr_re + hr_im * hr_im) * 3.814697265625e-06f);
            }
          u = fmaf (db, m_up[b], u);
          d = fmaf (db, m_dn[b], d);
        }
#pragma unroll
      for (int sh = 16; sh > 0; sh >>= 1)
        {
          u += __shfl_xor_sync (0xffffffffu, u, sh);
          d += __shfl_xor_sync (0xffffffffu, d, sh);
        }
      if (lane == 0)
        {
          // frames in digital silence are not counted (src/syncfinder.cc:573-580)
          const long long f_first = start * C, f_last = (start + kFrame) * C;
          const bool counted = !(f_last < wav_first || f_first > wav_last);
          out[(size_t) m * n_ent] = make_float2 (u, d);
          flag[(size_t) m * n_ent] = counted ? 1 : 0;
        }
      if (m + 1 >= n_valid)
        break;
      // ---- slide by 8 samples
#pragma unroll
      for (int b = 0; b < kSlideBins; b++)
        {
          float tr = rl_re[b], ti = rl_im[b];
#pragma unroll
          for (int j = 0; j < 8; j++)
            {
              tr = fmaf (dl[j], wr[b][j], tr);
              ti = fmaf (dl[j], wi[b][j], ti);
            }
          rl_re[b] = tr * rot_c[b] - ti * rot_s[b];
          rl_im[b] = tr * rot_s[b] + ti * rot_c[b];
          if (C == 2)
            {
              float sr = rr_re[b], si = rr_im[b];
#pragma unroll
              for (int j = 0; j < 8; j++)
                {
                  sr = fmaf (dr[j], wr[b][j], sr);
                  si = fmaf (dr[j], wi[b][j], si);
                }
              rr_re[b] = sr * rot_c[b] - si * rot_s[b];
              rr_im[b] = sr * rot_s[b] + si * rot_c[b];
            }
        }
    }
}

// per (candidate, offset, sync bit): add the per-frame sums in frame order, count the frames that were used
// -> the layout k_refine writes (out_ud / out_cnt / out_valid), so the host side is unchanged
__global__ void
k_refine_reduce (const float2 *__restrict__ ent_ud, const unsigned char *__restrict__ ent_flag, int n_cand, int n_ent,
                 const int *__restrict__ g_bit_off, int n_bits, const long long *__restrict__ cand_start, const int *__restrict__ cand_noff,
                 long long n_frames, int total_frame_count,
                 float *__restrict__ out_ud, int *__restrict__ out_cnt, unsigned char *__restrict__ out_valid)
{
  const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long) n_cand * kOffsets * n_bits)
    return;
  const int c = int (i / (kOffsets * n_bits)), o = int ((i / n_bits) % kOffsets), bit = int (i % n_bits);
  const long long fine = cand_start[c] + 8LL * o;
  const bool valid = o < cand_noff[c] && fine + (long long) total_frame_count * kFrame <= n_frames;
  if (bit == 0)
    out_valid[c * kOffsets + o] = valid ? 1 : 0;
  if (!valid)
    return;
  const float2 *ud = ent_ud + ((size_t) c * kOffsets + o) * n_ent;
  const unsigned char *fl = ent_flag + ((size_t) c * kOffsets + o) * n_ent;
  float umag = 0.f, dmag = 0.f;
  int cnt = 0;
  for (int e = g_bit_off[bit]; e < g_bit_off[bit + 1]; e++)
    if (fl[e])
      {
        const float2 v = ud[e];
        umag += v.x;
        dmag += v.y;
        cnt++;
      }
  const size_t ob = ((size_t) c * kOffsets + o) * n_bits + bit;
  out_ud[ob * 2] = umag;
  out_ud[ob * 2 + 1] = dmag;
  out_cnt[ob] = cnt;
}

} // namespace awm

namespace awm {

// ---- exact re-scoring of a few (candidate, offset) pairs picked by the sliding pass -------------------------------------------
// k_refine computes the same thing with one warp per (pair, sync bit) walking 85 frames one after the other; for a handful of
// pairs that is a long serial chain on a nearly empty GPU.  Here the transforms run in parallel (warp = one pair x one sync frame,
// time-domain window and arithmetic of frame_db_sum, i.e. of the reference's sync_fft) and only the additions stay serial:
// k_refine_exact_sum adds the stored band values of a bit in the reference's order (frames ascending, 30 up / 30 down bands each).
constexpr int kExactWarps = 8;

__global__ void __launch_bounds__ (kExactWarps * 32, 2)
k_refine_exact_fft (const float *__restrict__ pcm, long long n_frames, int C, const long long *__restrict__ pair_start, int n_pairs,
                    const awm_sync_entry *__restrict__ g_ent, int n_ent, float *__restrict__ vals /* [pair][entry][60] */,
                    const float2 *g_tw, const float *g_win)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, g_tw, g_win, kExactWarps);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float *sband = s.extra + w * 96;
  const long long job = (long long) blockIdx.x * kExactWarps + w;
  if (job >= (long long) n_pairs * n_ent)
    return;
  const int p = int (job / n_ent), e = int (job % n_ent);
  const awm_sync_entry *en = g_ent + e;
  const long long start = pair_start[p] + (long long) en->frame * kFrame;
  float acc[4];
  frame_db_sum (pcm, n_frames, C, start, s, lane, acc);
  bands_to_array (acc, lane, sband, 1);
  __syncwarp();
  float *o = vals + ((size_t) p * n_ent + e) * (2 * kUD);
  if (lane < kUD)
    {
      o[lane] = sband[en->up[lane]];
      o[kUD + lane] = sband[en->down[lane]];
    }
}

// One warp per (pair, sync bit, up / down): the 30 band values of every frame of the bit are first staged in shared memory by the
// whole warp (coalesced), then lane 0 adds them one after the other in the reference's order -- the chain of ~2550 dependent float
// additions is what this kernel's time consists of, the loads no longer sit between them.
constexpr int kExactSumWarps = 4;

__global__ void __launch_bounds__ (kExactSumWarps * 32)
k_refine_exact_sum (const float *__restrict__ vals, const long long *__restrict__ pair_start, int n_pairs, long long n_frames, int C,
                    const awm_sync_entry *__restrict__ g_ent, int n_ent, const int *__restrict__ g_bit_off, int n_bits, int total_frame_count,
                    long long wav_first, long long wav_last, int max_bit_frames,
                    float *__restrict__ out_ud /* [pair][n_bits][2] */, int *__restrict__ out_cnt, unsigned char *__restrict__ out_valid)
{
  extern __shared__ __align__ (16) unsigned char smem[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float *stage = reinterpret_cast<float *> (smem) + size_t (w) * max_bit_frames * kUD;
  const int i = blockIdx.x * kExactSumWarps + w;
  if (i >= n_pairs * n_bits * 2)
    return;
  const int p = i / (n_bits * 2), bit = (i / 2) % n_bits, which = i & 1;       // which: 0 = up bands, 1 = down bands
  const long long fine = pair_start[p];
  const bool valid = fine + (long long) total_frame_count * kFrame <= n_frames;
  if (bit == 0 && which == 0 && lane == 0)
    out_valid[p] = valid ? 1 : 0;
  if (!valid)
    return;
  const int e0 = g_bit_off[bit], e1 = g_bit_off[bit + 1];
  for (int k = lane; k < (e1 - e0) * kUD; k += 32)
    stage[k] = __ldg (vals + ((size_t) p * n_ent + e0 + k / kUD) * (2 * kUD) + which * kUD + k % kUD);
  __syncwarp();
  if (lane != 0)
    return;
  float mag = 0.f;
  int cnt = 0;
  for (int e = e0; e < e1; e++)
    {
      const long long start = fine + (long long) g_ent[e].frame * kFrame;
      const long long f_first = start * C, f_last = (start + kFrame) * C;
      if (f_last < wav_first || f_first > wav_last)        // frames in digital silence are not counted
        continue;
      const float *v = stage + (e - e0) * kUD;
#pragma unroll
      for (int k = 0; k < kUD; k++)
        mag = __fadd_rn (mag, v[k]);
      cnt++;
    }
  out_ud[((size_t) p * n_bits + bit) * 2 + which] = mag;
  if (which == 0)
    out_cnt[(size_t) p * n_bits + bit] = cnt;
}

} // namespace awm
