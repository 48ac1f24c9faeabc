// awm_speed.cuh -- kernels of the resampler and of the speed detection scan (sm_100a).
//
//   k_resample       windowed-sinc polyphase resampler, one thread per output frame.  Stands in for the
//                    zita-resampler calls of src/resample.cc:27-131 (process_resampler / resample /
//                    resample_ratio_truncate); zita itself is a third-party library that is not part of the reference
//                    tree, the filter definition used here is stated in DESIGN.md and in awm_b200.h.
//   k_speed_mags     SpeedSync::prepare_mags (src/wmspeed.cc:203-268): 512-point spectra of the half-rate clip at a
//                    hop of 128, channel-summed dB of bins 20..100, up/down sums per sync entry -> MagMatrix
//   k_speed_compare  SpeedSync::compare + compare_bits (src/wmspeed.cc:270-375): for one relative speed all 8908 start
//                    offsets are scored against three blocks of sync frames, the best |quality| is kept
#pragma once
#include "awm_fft.cuh"
#include "../../include/awm_b200.h"

namespace awm {

constexpr int kResamplePhases = 256;

struct ResampleJob
{
  const float *in;          // [n_in][C]
  float       *out;         // [n_out][C]
  long long    n_in, n_out;
  long long    n_stop;      // outputs whose centre lies at or beyond n_stop are 0 (where a stream with h frames of post-roll
                            // ends): n_in for resample(), "never" when the input is followed by more zeros
  double       step;        // input frames per output frame = 1 / ratio
  int          h;           // half filter length in input frames; 2h taps
  const float *coef;        // [2h][kResamplePhases + 1]: tap major, so that the lanes of a warp (same tap, different phase)
                            // gather inside one 1 KB row instead of touching 32 different rows
};

// out[n] = sum_j x[c - 2h + 2 + j] * ((1-a) coef[p][j] + a coef[p+1][j]),  t = (h-1) + n step, c = floor t,
// (p, a) = integer / fractional part of 256 (t - c); x is zero outside [0, n_in).  Float products and sums are kept
// separate and in tap order, t is evaluated in closed form in double: a sequential implementation that does the same
// gets the same bits.
template<int C> __global__ void __launch_bounds__ (256)
k_resample (const ResampleJob *__restrict__ jobs, int c_dyn)
{
  const ResampleJob J = jobs[blockIdx.y];
  const int CH = C > 0 ? C : c_dyn;
  const int h = J.h, taps = 2 * h;
  for (long long n = (long long) blockIdx.x * blockDim.x + threadIdx.x; n < J.n_out; n += (long long) gridDim.x * blockDim.x)
    {
      const double t = __dadd_rn (double (h - 1), __dmul_rn (double (n), J.step));
      const double fl = floor (t);
      const long long c = (long long) fl;
      float *o = J.out + n * CH;
      if (c > J.n_stop + h - 2)                  // taps would run past the post-roll: a streaming resampler stops here
        {
          for (int ch = 0; ch < CH; ch++)
            o[ch] = 0.0f;
          continue;
        }
      const double frac = __dmul_rn (__dsub_rn (t, fl), double (kResamplePhases));
      const int p = int (frac);
      const float a = float (__dsub_rn (frac, double (p))), b = __fsub_rn (1.0f, a);
      const float *c0 = J.coef + p, *c1 = c0 + 1;
      constexpr int RS = kResamplePhases + 1;        // row stride of the tap-major table
      const long long i0 = c - 2LL * h + 2;
      if (C == 2)
        {
          float s0 = 0.0f, s1 = 0.0f;
          const float2 *x2 = reinterpret_cast<const float2 *> (J.in);
          for (int j = 0; j < taps; j++)
            {
              const long long i = i0 + j;
              const float w = __fadd_rn (__fmul_rn (b, __ldg (c0 + j * RS)), __fmul_rn (a, __ldg (c1 + j * RS)));
              const float2 x = (i >= 0 && i < J.n_in) ? __ldg (x2 + i) : make_float2 (0.0f, 0.0f);
              s0 = __fadd_rn (s0, __fmul_rn (x.x, w));
              s1 = __fadd_rn (s1, __fmul_rn (x.y, w));
            }
          reinterpret_cast<float2 *> (J.out)[n] = make_float2 (s0, s1);
        }
      else
        {
          for (int ch = 0; ch < CH; ch++)
            {
              float s = 0.0f;
              for (int j = 0; j < taps; j++)
                {
                  const long long i = i0 + j;
                  const float w = __fadd_rn (__fmul_rn (b, __ldg (c0 + j * RS)), __fmul_rn (a, __ldg (c1 + j * RS)));
                  const float x = (i >= 0 && i < J.n_in) ? __ldg (J.in + i * CH + ch) : 0.0f;
                  s = __fadd_rn (s, __fmul_rn (x, w));
                }
              o[ch] = s;
            }
        }
    }
}

// float -> 16 bit PCM exactly as the reference writes it: float_to_int_clip<32> (src/rawconverter.hh:34-50), the 16 most
// significant bits kept (src/sfoutputstream.cc:148-155).  Reading is k_wav_to_f32<WAV_S16> (awm_wav_decode.cuh).
__device__ __forceinline__ int16_t
f32_to_s16 (float f)
{
  const float snorm = __fmul_rn (f, 2147483648.0f);
  int v;
  if (snorm >= 2147483648.0f)            // max_value = float (2^31 - 1) = 2^31
    v = 0x7fffffff;
  else if (snorm <= -2147483648.0f)
    v = int (0x80000000u);
  else
    v = int (snorm);                     // truncation toward zero
  return int16_t (v >> 16);
}

__global__ void
k_f32_to_s16 (const float *__restrict__ in, int16_t *__restrict__ out, long long n)
{
  const long long i = ((long long) blockIdx.x * blockDim.x + threadIdx.x) * 2;
  if (i + 1 < n)
    {
      const float2 v = *reinterpret_cast<const float2 *> (in + i);
      short2 o;
      o.x = f32_to_s16 (v.x);
      o.y = f32_to_s16 (v.y);
      *reinterpret_cast<short2 *> (out + i) = o;
    }
  else if (i < n)
    out[i] = f32_to_s16 (in[i]);
}

// dst[k] = src[idx[k]]: the sparse sample subset get_clip_locations hashes (src/wmspeed.cc:538-543) when the PCM lives in device memory
__global__ void
k_gather (const float *__restrict__ src, const unsigned long long *__restrict__ idx, long long n, float *__restrict__ dst)
{
  const long long k = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n)
    dst[k] = __ldg (src + idx[k]);
}

// out[i] = orig[i] + wm[i] for the frames the add loop emits (src/wmadd.cc:548-566 with a WatermarkResampler): orig is zero
// beyond n_in; per limiter block the peak of |out| (only peaks above the ceiling matter, Limiter::block_max starts at the
// ceiling) and the --snr sums.  Values are stored for i < n_in only, the limiter rescales them in place afterwards.
__global__ void __launch_bounds__ (256)
k_mix_peaks (const float *__restrict__ orig, long long n_in, const float *__restrict__ wm, long long n_emit, int C, float *__restrict__ out,
             int limiter_block, float ceiling, unsigned *__restrict__ peaks, double *__restrict__ snr)
{
  const long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  double sd = 0, ss = 0;
  if (i < n_emit)
    {
      float mx = 0.f;
      for (int c = 0; c < C; c++)
        {
          const float o = i < n_in ? __ldg (orig + i * C + c) : 0.f;
          const float w = __ldg (wm + i * C + c);
          const float y = __fadd_rn (w, o);
          if (i < n_in)
            out[i * C + c] = y;
          mx = fmaxf (mx, fabsf (y));
          sd += double (w) * double (w);
          ss += double (o) * double (o);
        }
      if (limiter_block > 0 && mx > ceiling)
        atomicMax (peaks + i / limiter_block, __float_as_uint (mx));
    }
  if (snr)
    {
      for (int d = 16; d > 0; d >>= 1)
        {
          sd += __shfl_xor_sync (0xffffffffu, sd, d);
          ss += __shfl_xor_sync (0xffffffffu, ss, d);
        }
      if ((threadIdx.x & 31) == 0 && (sd != 0 || ss != 0))
        {
          atomicAdd (snr, sd);
          atomicAdd (snr + 1, ss);
        }
    }
}

// ---------------------------------------------------------------------------------------------- speed scan

constexpr int kSpeedFrame = 512;           // Params::frame_size / 2          (src/wmspeed.cc:209)
constexpr int kSpeedHop = 128;             // Params::sync_search_step / 2    (src/wmspeed.cc:210)
constexpr int kMagWarps = 8;
constexpr int kMagRows = 2 * kMagWarps;    // rows of the MagMatrix one CTA produces
constexpr size_t kMagSmemBytes = (size_t (kMagWarps) * kWarpFftSmemFloats + kBands * kMagRows) * sizeof (float);

struct MagJob
{
  const float *sub;      // half-rate clip [n_sub][C]
  long long    n_sub;
  int          rows;     // positions pos = 128 r with pos + 512 < n_sub
  float2      *mags;     // [n_entries][rows] (umag, dmag): MagMatrix is column major (src/wmspeed.cc:75-79)
};

// dB of (are + i aim) +- (bre + i bim), halved: the two 512-point spectra that were interleaved into one 1024-point FFT
__device__ __forceinline__ void
split_rows_db (float are, float aim, float bre, float bim, float& db_even, float& db_odd)
{
  db_even = db_from_complex (0.5f * (are + bre), 0.5f * (aim + bim), -96.0f);
  db_odd  = db_from_complex (0.5f * (are - bre), 0.5f * (aim - bim), -96.0f);
}

// One warp transforms two rows at once: z[2m] = row r, z[2m+1] = row r+1 (each windowed, 512 samples, left + i right).
// With Z = FFT_1024 (z):  X_r[k] = (Z[k] + Z[k+512]) / 2,  X_{r+1}[k] = (Z[k] - Z[k+512]) / (2 W_1024^k); only |X|
// is needed, so the twiddle drops out.  Bins 20..100 live in registers k2 = 0..3 (k = lane + 32 k2), their partners
// k + 512 in k2 + 16.
template<int K2> __device__ __forceinline__ void
speed_db_k2 (const float (&re)[32], const float (&im)[32], int lane, bool second_channel, unsigned zero, float& acc_even, float& acc_odd)
{
  float a0r, a0i, b0r, b0i, a1r, a1i, b1r, b1i;
  unpack_pair<K2> (re, im, lane, a0r, a0i, b0r, b0i, zero);
  unpack_pair<K2 + 16> (re, im, lane, a1r, a1i, b1r, b1i, zero);
  float e, o;
  split_rows_db (a0r, a0i, a1r, a1i, e, o);
  acc_even = __fadd_rn (acc_even, e);
  acc_odd = __fadd_rn (acc_odd, o);
  if (second_channel)
    {
      split_rows_db (b0r, b0i, b1r, b1i, e, o);
      acc_even = __fadd_rn (acc_even, e);
      acc_odd = __fadd_rn (acc_odd, o);
    }
}

__global__ void __launch_bounds__ (kMagWarps * 32)
k_speed_mags (const MagJob *__restrict__ jobs, int C, const awm_sync_entry *__restrict__ ent, int n_ent,
              const float2 *__restrict__ g_tw, const float *__restrict__ win512)
{
  extern __shared__ __align__ (16) float sm_speed[];
  float *xbuf_all = sm_speed;
  float *db = sm_speed + kMagWarps * kWarpFftSmemFloats;        // [band][kMagRows]
  const MagJob J = jobs[blockIdx.y];
  const int row0 = blockIdx.x * kMagRows;
  if (row0 >= J.rows)
    return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float *xbuf = xbuf_all + warp * kWarpFftSmemFloats;

  // ---- phase 1: spectra of rows row0 + 2 warp, + 1
  {
    const int my_row = row0 + 2 * warp + (lane & 1);
    const bool row_ok = my_row < J.rows;
    const long long base = (long long) my_row * kSpeedHop;
    float acc_e[4] = { 0.f, 0.f, 0.f, 0.f }, acc_o[4] = { 0.f, 0.f, 0.f, 0.f };     // fft_out_db.fill (0), src/wmspeed.cc:233
    for (int c0 = 0; c0 < C; c0 += 2)
      {
        const bool two = c0 + 1 < C;
        float re[32], im[32];
#pragma unroll
        for (int j = 0; j < 32; j++)
          {
            const int m = 16 * j + (lane >> 1);
            float xr = 0.f, xi = 0.f;
            if (row_ok)
              {
                const float w = __ldg (win512 + m);
                const float *s = J.sub + (base + m) * C + c0;
                xr = __fmul_rn (__ldg (s), w);
                if (two)
                  xi = __fmul_rn (__ldg (s + 1), w);
              }
            re[j] = xr;
            im[j] = xi;
          }
        const unsigned zero = pair_zero_mask (re, im);
        fft1024_warp (re, im, g_tw, xbuf, lane);
        speed_db_k2<0> (re, im, lane, two, zero, acc_e[0], acc_o[0]);
        speed_db_k2<1> (re, im, lane, two, zero, acc_e[1], acc_o[1]);
        speed_db_k2<2> (re, im, lane, two, zero, acc_e[2], acc_o[2]);
        speed_db_k2<3> (re, im, lane, two, zero, acc_e[3], acc_o[3]);
      }
#pragma unroll
    for (int k2 = 0; k2 < 4; k2++)
      {
        const int k = lane + 32 * k2;
        if (k >= kMinBand && k <= kMaxBand)
          {
            db[(k - kMinBand) * kMagRows + 2 * warp] = acc_e[k2];
            db[(k - kMinBand) * kMagRows + 2 * warp + 1] = acc_o[k2];
          }
      }
  }
  __syncthreads();

  // ---- phase 2: up / down sums of every sync entry for the 16 rows (src/wmspeed.cc:251-262), summed in list order
  for (int e = threadIdx.x; e < n_ent; e += blockDim.x)
    {
      float um[kMagRows], dm[kMagRows];
#pragma unroll
      for (int r = 0; r < kMagRows; r++)
        um[r] = dm[r] = 0.f;
      const awm_sync_entry *E = ent + e;
      for (int i = 0; i < kUD; i++)
        {
          const float4 *pu = reinterpret_cast<const float4 *> (db + int (E->up[i]) * kMagRows);
          const float4 *pd = reinterpret_cast<const float4 *> (db + int (E->down[i]) * kMagRows);
#pragma unroll
          for (int q = 0; q < kMagRows / 4; q++)
            {
              const float4 u = pu[q], d = pd[q];
              um[4 * q + 0] = __fadd_rn (um[4 * q + 0], u.x); um[4 * q + 1] = __fadd_rn (um[4 * q + 1], u.y);
              um[4 * q + 2] = __fadd_rn (um[4 * q + 2], u.z); um[4 * q + 3] = __fadd_rn (um[4 * q + 3], u.w);
              dm[4 * q + 0] = __fadd_rn (dm[4 * q + 0], d.x); dm[4 * q + 1] = __fadd_rn (dm[4 * q + 1], d.y);
              dm[4 * q + 2] = __fadd_rn (dm[4 * q + 2], d.z); dm[4 * q + 3] = __fadd_rn (dm[4 * q + 3], d.w);
            }
        }
      float2 *out = J.mags + (size_t) e * J.rows + row0;
#pragma unroll
      for (int r = 0; r < kMagRows; r++)
        if (row0 + r < J.rows)
          out[r] = make_float2 (um[r], dm[r]);
    }
}

struct CmpJob
{
  const float2 *mags;
  int           rows;
  double        inv;         // 1 / relative_speed
  double        off_scale;   // 65536 / relative_speed
};

constexpr int kCmpMaxEntries = 1024;

// thread = one start offset (CmpState, src/wmspeed.cc:118-122).  The reference walks the frame-sorted entry list once per
// block and scatters into six per-bit accumulators; the per-bit sums only depend on the order inside a bit, so here each
// bit is summed on its own (entries are stored bit major, frame sorted inside a bit: the layout of awm_set_sync_tables).
// The begin / end iterators of compare_bits are the index tests s >= 0 and (s >> 16) < rows: offsets and frame offsets
// both grow monotonically.
__global__ void __launch_bounds__ (256)
k_speed_compare (const CmpJob *__restrict__ jobs, const awm_sync_entry *__restrict__ ent, const int *__restrict__ bit_off, int n_bits,
                 int n_ent, int frames_per_block, int pad_start, double norm_div, unsigned long long *__restrict__ best)
{
  __shared__ int fo[3 * kCmpMaxEntries];
  const CmpJob J = jobs[blockIdx.y];
  for (int idx = threadIdx.x; idx < 3 * n_ent; idx += blockDim.x)
    {
      const int B = idx / n_ent, e = idx - B * n_ent;
      const int v = (B * frames_per_block + int (ent[e].frame)) * 4;             // steps_per_frame = 4
      fo[idx] = int (__dmul_rn (__dadd_rn (__dmul_rn (double (v), J.inv), 0.5), 65536.0));   // src/wmspeed.cc:280
    }
  __syncthreads();
  const int o = blockIdx.x * blockDim.x + threadIdx.x;
  double quality = 0;
  if (o < pad_start)
    {
      const int offset = int (__dmul_rn (double (o - pad_start), J.off_scale));   // src/wmspeed.cc:341
      double sync_quality = 0;
      int bit_count = 0;
      for (int bit = 0; bit < n_bits; bit++)
        {
          float umag = 0.f, dmag = 0.f;
          int count = 0;
          const int e0 = bit_off[bit], e1 = bit_off[bit + 1];
#pragma unroll
          for (int B = 0; B < 3; B++)
            {
              const int *f = fo + B * n_ent;
              for (int e = e0; e < e1; e++)
                {
                  const int s = offset + f[e];
                  const int index = s >> 16;
                  if (s >= 0 && index < J.rows)
                    {
                      const float2 m = __ldg (J.mags + (size_t) e * J.rows + index);
                      if (B & 1)
                        {
                          umag = __fadd_rn (umag, m.y);
                          dmag = __fadd_rn (dmag, m.x);
                        }
                      else
                        {
                          umag = __fadd_rn (umag, m.x);
                          dmag = __fadd_rn (dmag, m.y);
                        }
                      count++;
                    }
                }
            }
          double raw_bit;                                        // SyncFinder::bit_quality, src/syncfinder.cc:94-114
          if (umag == 0 || dmag == 0)
            raw_bit = 0;
          else if (umag < dmag)
            raw_bit = __fsub_rn (1.0f, __fdiv_rn (umag, dmag));
          else
            raw_bit = __fsub_rn (__fdiv_rn (dmag, umag), 1.0f);
          sync_quality += ((bit & 1) ? raw_bit : -raw_bit) * count;
          bit_count += count;
        }
      if (bit_count)
        quality = fabs (sync_quality / bit_count / norm_div / 2.9);
    }
  // best score of the job: maximum over offsets (non-negative doubles order like their bit patterns)
  for (int d = 16; d > 0; d >>= 1)
    quality = fmax (quality, __shfl_xor_sync (0xffffffffu, quality, d));
  if ((threadIdx.x & 31) == 0 && quality > 0)
    atomicMax (best + blockIdx.y, (unsigned long long) __double_as_longlong (quality));
}

} // namespace awm
