// awm_fft.cuh -- warp-resident 1024-point complex FFT for sm_100a.
//
// Replaces FFTProcessor / FFTW (reference src/fft.hh:25-44, src/fft.cc:51-118): the
// reference runs one r2c/c2r plan per channel per frame on the CPU; here one warp
// transforms one *pair* of real sequences (a + i*b, e.g. left + i*right of a stereo
// frame) as a single 1024-point complex FFT held entirely in registers:
//
//   n = 32*j + t   (t = lane, j = register)      1024 = 32 x 32 Cooley-Tukey
//   pass 1: per-lane 32-point DIF FFT over j      -> Y_t[k1]
//   twiddle W_1024^(t*k1), transpose through shared memory (padded, conflict free)
//   pass 2: per-lane 32-point DIF FFT over t      -> X[k1 + 32*k2], lane = k1
//
// After fft1024_warp() register i of lane k1 holds X[k1 + 32*brev5(i)].
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace awm {

constexpr int kFrame = 1024;          // Params::frame_size (src/wmcommon.hh:36)
constexpr int kMinBand = 20;          // src/wmcommon.hh:40
constexpr int kMaxBand = 100;         // src/wmcommon.hh:39
constexpr int kBands = kMaxBand - kMinBand + 1;
constexpr int kUD = 30;               // Params::bands_per_frame

__host__ __device__ constexpr int brev5 (int i)
{
  return ((i & 1) << 4) | ((i & 2) << 2) | (i & 4) | ((i & 8) >> 2) | ((i & 16) >> 4);
}

// cos / sin (2 pi i / 32), i = 0..8, as literals so that unrolled butterflies use immediates
__host__ __device__ constexpr float cos32 (int i)
{
  return i == 0 ? 1.0f : i == 1 ? 0.98078528040323043f : i == 2 ? 0.92387953251128674f : i == 3 ? 0.83146961230254524f
       : i == 4 ? 0.70710678118654752f : i == 5 ? 0.55557023301960218f : i == 6 ? 0.38268343236508978f
       : i == 7 ? 0.19509032201612825f : 0.0f;
}
__host__ __device__ constexpr float w32_re (int i)   // Re exp(-2 pi i idx/32), idx = 0..15
{
  return i <= 8 ? cos32 (i) : -cos32 (16 - i);
}
__host__ __device__ constexpr float w32_im (int i)   // Im exp(-2 pi i idx/32) = -sin
{
  return i <= 8 ? -cos32 (8 - i) : -cos32 (i - 8);
}

// (tr + i ti) * W32^IDX  with the trivial cases spelled out
template<int IDX> __device__ __forceinline__ void
twiddle32 (float tr, float ti, float& orr, float& oi)
{
  if (IDX == 0)       { orr = tr; oi = ti; }
  else if (IDX == 8)  { orr = ti; oi = -tr; }
  else if (IDX == 4)  { const float r = 0.70710678118654752f; orr = (tr + ti) * r; oi = (ti - tr) * r; }
  else if (IDX == 12) { const float r = 0.70710678118654752f; orr = (ti - tr) * r; oi = -(tr + ti) * r; }
  else
    {
      /* one multiply + one fused multiply-add per component, spelled out: which of the two products gets fused is then the same
       * in every kernel this is inlined into (left to the compiler it depends on the surrounding code, and two kernels that
       * should agree bit for bit differ in the last digit) */
      const float c = w32_re (IDX), s = w32_im (IDX);
      orr = __fmaf_rn (tr, c, -__fmul_rn (ti, s));
      oi  = __fmaf_rn (tr, s, __fmul_rn (ti, c));
    }
}

template<int LEN, int BASE, int K> struct DifK
{
  static __device__ __forceinline__ void run (float (&re)[32], float (&im)[32])
  {
    constexpr int HALF = LEN / 2;
    constexpr int i0 = BASE + K, i1 = i0 + HALF;
    const float ar = re[i0], ai = im[i0], br = re[i1], bi = im[i1];
    re[i0] = ar + br;
    im[i0] = ai + bi;
    twiddle32<K * (32 / LEN)> (ar - br, ai - bi, re[i1], im[i1]);
    if constexpr (K + 1 < HALF)
      DifK<LEN, BASE, K + 1>::run (re, im);
    else if constexpr (BASE + LEN < 32)
      DifK<LEN, BASE + LEN, 0>::run (re, im);
  }
};

// in-register 32-point DIF FFT, forward sign; output index i holds bin brev5(i)
__device__ __forceinline__ void
fft32_dif (float (&re)[32], float (&im)[32])
{
  DifK<32, 0, 0>::run (re, im);
  DifK<16, 0, 0>::run (re, im);
  DifK<8, 0, 0>::run (re, im);
  DifK<4, 0, 0>::run (re, im);
  DifK<2, 0, 0>::run (re, im);
}

constexpr int kWarpFftSmemFloats = 2 * 32 * 33;     // 32 x 33 float2, row stride 33 (bank-conflict free)

// 1024-point forward FFT of the warp's 32x32 register tile.
//   in : re[j], im[j] = z[32*j + lane]
//   out: re[i], im[i] = Z[lane + 32*brev5(i)]
//   tw : shared copy of exp(-2 pi i k1 t / 1024) at [k1*32 + t]
//   xbuf: this warp's transpose buffer (kWarpFftSmemFloats floats)
// `after_transpose` runs once the warp has read everything back from its transpose buffer, i.e. from the moment xbuf is free
// again: k_stft_mags_tc starts the bulk copy of the warp's next frame into it there, under the second pass of butterflies.
template<class Hook> __device__ __forceinline__ void
fft1024_warp (float (&re)[32], float (&im)[32], const float2 *tw, float *xbuf, int lane, Hook after_transpose)
{
  fft32_dif (re, im);
  float2 *xb = reinterpret_cast<float2 *> (xbuf);        // [32][33] complex, row stride 33: 64-bit accesses stay conflict free
#pragma unroll
  for (int i = 0; i < 32; i++)
    {
      const int k1 = brev5 (i);
      const float2 w = tw[k1 * 32 + lane];
      xb[k1 * 33 + lane] = make_float2 (__fmaf_rn (re[i], w.x, -__fmul_rn (im[i], w.y)), __fmaf_rn (re[i], w.y, __fmul_rn (im[i], w.x)));
    }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < 32; t++)
    {
      const float2 v = xb[lane * 33 + t];
      re[t] = v.x;
      im[t] = v.y;
    }
  __syncwarp();
  after_transpose();
  fft32_dif (re, im);
}

__device__ __forceinline__ void
fft1024_warp (float (&re)[32], float (&im)[32], const float2 *tw, float *xbuf, int lane)
{
  fft1024_warp (re, im, tw, xbuf, lane, [] {});
}

// Which of the two real inputs packed into (re, im) -- before the transform -- are zero in every sample of the warp: bit 0 the real
// part a, bit 1 the imaginary part b.  ORing the bit patterns and dropping the sign bit counts -0.0 as zero.
__device__ __forceinline__ unsigned
pair_zero_mask (const float (&re)[32], const float (&im)[32])
{
  unsigned oa = 0, ob = 0;
#pragma unroll
  for (int j = 0; j < 32; j++)
    {
      oa |= __float_as_uint (re[j]);
      ob |= __float_as_uint (im[j]);
    }
  return (__all_sync (0xffffffffu, (oa << 1) == 0) ? 1u : 0u) | (__all_sync (0xffffffffu, (ob << 1) == 0) ? 2u : 0u);
}

// Split the packed spectrum Z = FFT (a + i b) into the spectra of the two real inputs for
// bin k = lane + 32*K2:   A[k] = (Z[k] + conj Z[N-k]) / 2,   B[k] = (Z[k] - conj Z[N-k]) / (2i)
// Z[N-k] lives in lane (32-lane)&31 (register for k2' = 31-K2; lane 0 keeps k2' = (32-K2)&31).
// `zero` (pair_zero_mask of the input): an input that is zero in every sample has an exactly zero spectrum -- the reference then
// gets -96 dB in every bin (db_from_complex) -- while the formula above would return the rounding error of the other input's
// transform (the float FFT of a real input is not exactly Hermitian) at float rounding level of that input's magnitude.
template<int K2> __device__ __forceinline__ void
unpack_pair (const float (&re)[32], const float (&im)[32], int lane, float& ar, float& ai, float& br, float& bi, unsigned zero = 0)
{
  constexpr int I = brev5 (K2 & 31), IP = brev5 ((31 - K2) & 31), IP0 = brev5 ((32 - K2) & 31);
  const float sr = (lane == 0) ? re[IP0] : re[IP];
  const float si = (lane == 0) ? im[IP0] : im[IP];
  const int src = (32 - lane) & 31;
  const float pr = __shfl_sync (0xffffffffu, sr, src);
  const float pi = __shfl_sync (0xffffffffu, si, src);
  const float zr = re[I], zi = im[I];
  ar = 0.5f * (zr + pr);
  ai = 0.5f * (zi - pi);
  br = 0.5f * (zi + pi);
  bi = -0.5f * (zr - pr);
  if (zero & 1u)
    ar = ai = 0.f;
  if (zero & 2u)
    br = bi = 0.f;
}

// db_from_complex (reference src/wmcommon.hh:204-224)
__device__ __forceinline__ float
db_from_complex (float re, float im, float min_db)
{
  const float abs2 = __fmaf_rn (re, re, __fmul_rn (im, im));
  return abs2 > 0.0f ? log2f (abs2) * 3.01029995663981f : min_db;
}

// the same from the squared magnitude
__device__ __forceinline__ float
db_from_complex_abs2 (float abs2)
{
  return abs2 > 0.0f ? log2f (abs2) * 3.01029995663981f : -96.0f;
}

} // namespace awm
