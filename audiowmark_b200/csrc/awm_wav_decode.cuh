// awm_wav_decode.cuh -- stored WAV sample bytes -> the float samples the pipeline works on (sm_100a).
//
//   k_wav_to_f32<T>  one kernel for every sample format a WAV input of `get` can hold: unsigned 8 bit, signed 16 / 24 / 32 bit
//                    and float 32 / 64 bit, all little endian.  The arithmetic is RawConverter::from_raw's (host/awm_streams.cc,
//                    src/rawconverter.cc): an integer sample is left justified to 32 bits (8 bit: offset by 2^31 first) and
//                    multiplied by 2^-31 in float; float32 is taken bit for bit; float64 is rounded to float like a cast on
//                    x86-64 (NaN payloads truncated, quiet bit set).  So the device copy is bit-identical to converting on
//                    the host, and only the stored bytes cross PCIe (24 bit audio: 3/4 of the float bytes, 16 bit: 1/2).
//
// A thread decodes four samples from 4 * bytes-per-sample bytes, read as aligned 32-bit words (24 bit: 12 bytes = three words
// hold four samples).  When the input does not start on a 16-byte boundary the words are assembled with funnel shifts from the
// aligned words around them; a word that holds at least one byte of the input is never outside its allocation.  The last
// n % 4 samples are read byte by byte.
#pragma once
#include <stdint.h>

namespace awm {

enum WavSampleType { WAV_U8 = 0, WAV_S16, WAV_S24, WAV_S32, WAV_F32, WAV_F64 };

template<int T> struct WavBytes;
template<> struct WavBytes<WAV_U8>  { static constexpr int n = 1; };
template<> struct WavBytes<WAV_S16> { static constexpr int n = 2; };
template<> struct WavBytes<WAV_S24> { static constexpr int n = 3; };
template<> struct WavBytes<WAV_S32> { static constexpr int n = 4; };
template<> struct WavBytes<WAV_F32> { static constexpr int n = 4; };
template<> struct WavBytes<WAV_F64> { static constexpr int n = 8; };

/* left-justified 32 bit sample -> float: int32 * 2^-31 (src/rawconverter.cc; exact for up to 24 significant bits) */
__device__ __forceinline__ float
wav_int_to_f32 (uint32_t s)
{
  return __fmul_rn (__int2float_rn (int (s)), 4.656612873077392578125e-10f);
}

/* double -> float as the host's cast rounds it (cvtsd2ss): round to nearest, denormals kept; a NaN keeps its sign and the top 23
 * bits of its payload and becomes quiet.  The NaN case is spelled out so that it does not depend on what the device's conversion
 * does with payloads. */
__device__ __forceinline__ float
wav_f64_to_f32 (uint32_t lo, uint32_t hi)
{
  if ((hi & 0x7ff00000u) == 0x7ff00000u && ((hi & 0xfffffu) | lo))
    return __uint_as_float ((hi & 0x80000000u) | 0x7fc00000u | ((hi & 0xfffffu) << 3) | (lo >> 29));
  return __double2float_rn (__hiloint2double (int (hi), int (lo)));
}

/* four samples from the 4 * WavBytes<T>::n bytes in w[] (little endian words) */
template<int T> __device__ __forceinline__ void
wav_decode4 (const uint32_t *w, float *f)
{
  if constexpr (T == WAV_U8)
    {
      for (int j = 0; j < 4; j++)
        f[j] = wav_int_to_f32 (((w[0] >> (8 * j)) << 24) ^ 0x80000000u);
    }
  else if constexpr (T == WAV_S16)
    {
      f[0] = wav_int_to_f32 (w[0] << 16);
      f[1] = wav_int_to_f32 (w[0] & 0xffff0000u);
      f[2] = wav_int_to_f32 (w[1] << 16);
      f[3] = wav_int_to_f32 (w[1] & 0xffff0000u);
    }
  else if constexpr (T == WAV_S24)
    {
      /* bytes b0..b11 = w0 w1 w2; sample j = bytes 3j .. 3j+2, shifted to the top of the word */
      f[0] = wav_int_to_f32 (w[0] << 8);
      f[1] = wav_int_to_f32 ((w[1] << 16) | ((w[0] >> 24) << 8));
      f[2] = wav_int_to_f32 ((w[2] << 24) | ((w[1] >> 16) << 8));
      f[3] = wav_int_to_f32 (w[2] & 0xffffff00u);
    }
  else if constexpr (T == WAV_S32)
    {
      for (int j = 0; j < 4; j++)
        f[j] = wav_int_to_f32 (w[j]);
    }
  else if constexpr (T == WAV_F32)
    {
      for (int j = 0; j < 4; j++)
        f[j] = __uint_as_float (w[j]);
    }
  else
    {
      for (int j = 0; j < 4; j++)
        f[j] = wav_f64_to_f32 (w[2 * j], w[2 * j + 1]);
    }
}

/* one sample from its bytes (any alignment): the tail of the kernel */
template<int T> __device__ __forceinline__ float
wav_decode1 (const unsigned char *b)
{
  constexpr int B = WavBytes<T>::n;
  uint32_t w[2] = { 0, 0 };
  for (int k = 0; k < B; k++)
    w[k / 4] |= uint32_t (b[k]) << (8 * (k % 4));
  if constexpr (T == WAV_F32)
    return __uint_as_float (w[0]);
  else if constexpr (T == WAV_F64)
    return wav_f64_to_f32 (w[0], w[1]);
  else
    {
      uint32_t s = w[0] << (32 - 8 * B);
      if constexpr (T == WAV_U8)
        s ^= 0x80000000u;
      return wav_int_to_f32 (s);
    }
}

/* in: n samples of type T starting at any byte address; out: n floats (any 4-byte aligned address) */
template<int T>
__global__ void __launch_bounds__ (256)
k_wav_to_f32 (const unsigned char *__restrict__ in, float *__restrict__ out, long long n)
{
  constexpr int B = WavBytes<T>::n;                 // words per group of four samples
  const long long g = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  const long long i0 = g * 4;
  if (i0 + 4 <= n)
    {
      uint32_t w[B];
      const unsigned mis = unsigned (reinterpret_cast<uintptr_t> (in) & 15);
      if (mis == 0)
        {
          const uint32_t *p = reinterpret_cast<const uint32_t *> (in) + g * B;
          if constexpr (B == 1)
            w[0] = __ldg (p);
          else if constexpr (B == 2)
            {
              const uint2 v = __ldg (reinterpret_cast<const uint2 *> (p));
              w[0] = v.x; w[1] = v.y;
            }
          else if constexpr (B == 4 || B == 8)
            {
              for (int q = 0; q < B / 4; q++)
                {
                  const uint4 v = __ldg (reinterpret_cast<const uint4 *> (p) + q);
                  w[4 * q] = v.x; w[4 * q + 1] = v.y; w[4 * q + 2] = v.z; w[4 * q + 3] = v.w;
                }
            }
          else
            for (int k = 0; k < B; k++)
              w[k] = __ldg (p + k);
        }
      else
        {
          const uint32_t *a = reinterpret_cast<const uint32_t *> (in - (mis & 3)) + g * B;
          const unsigned shift = 8 * (mis & 3);
          uint32_t x[B + 1];
          for (int k = 0; k < B; k++)
            x[k] = __ldg (a + k);
          x[B] = shift ? __ldg (a + B) : 0;
          for (int k = 0; k < B; k++)
            w[k] = __funnelshift_r (x[k], x[k + 1], shift);
        }
      float f[4];
      wav_decode4<T> (w, f);
      if ((reinterpret_cast<uintptr_t> (out) & 15) == 0)
        *reinterpret_cast<float4 *> (out + i0) = make_float4 (f[0], f[1], f[2], f[3]);
      else
        for (int j = 0; j < 4; j++)
          out[i0 + j] = f[j];
    }
  else
    for (long long i = i0; i < n; i++)
      out[i] = wav_decode1<T> (in + i * B);
}

} // namespace awm
