// awm_approx_tc.cuh -- k_stft_mags_tc: SyncFinder::sync_fft for the four 256-sample shifts (src/syncfinder.cc:560-657) plus the
// inner sums of sync_decode (:116-153) as ONE persistent, warp-specialised Blackwell kernel.
//
// What it computes is what k_stft_mags (awm_approx_mags.cuh) computes: for every frame f of a shift the channel-summed band dB
// values dB[f][0..80], and from them, for every sync entry e (a sync frame with 30 "up" and 30 "down" bands),
//     U_e(f) = sum_{u in up(e)} dB[f][u],   D_e(f) = sum_{d in down(e)} dB[f][d]      -> mags[shift][e][f] = (U, D)
// The second step is the contraction  [128 frames x 96 bands] . [96 bands x 2 n_ent 0/1 columns].  On the fp32 pipes it costs
// 30 600 shared-memory reads + adds per frame and bounded the old kernel (2/3 of its time, shared-memory bandwidth).  Here it runs
// on the 5th generation tensor cores:
//   * A operand = the dB tile, written by the FFT warps straight into the K-major operand layout (awm_tc.cuh) as TWO fp16 terms
//     hi = fp16 (v), lo = fp16 (v - hi): |v| < 256, so hi + lo carries v to 2^-16 absolute -- the resolution fp32 itself has there;
//     every product with a 0/1 mask element is exact, accumulation is fp32 in tensor memory
//   * B operand = the 0/1 masks of 128 entries (256 columns: U and D of an entry side by side), prepared once per key on the host
//     in operand layout and fetched chunk by chunk with the bulk-copy engine (TMA, cp.async.bulk -> mbarrier complete_tx)
//   * D = 128 x 256 fp32 in TMEM, double buffered (2 x 256 of the 512 columns): tcgen05.mma of chunk g + 1 runs while the
//     epilogue warps drain chunk g with tcgen05.ld and write coalesced float2 rows of `mags`
// Warp roles (one CTA per SM, CTAs walk the (frame tile, shift) list with stride gridDim.x):
//   warps 0 .. F-1     FFT: frame (PCM prefetched by TMA into the warp's transpose buffer) -> packed 1024-point FFT -> dB ->
//                      fp16 hi/lo into A[buf]                                                     (a_empty -> a_full)
//   warps F .. F+3     epilogue: TMEM -> registers -> global                                      (tmem_full -> tmem_empty)
//   warp  F+4, lane 0  TMA + MMA issue: B chunk load, 2 x 6 tcgen05.mma, commits                  (a_full, b_full, tmem_empty -> ...)
// All hand-offs are mbarriers; the FFT of tile i + 1 overlaps the MMAs and the epilogue of tile i.
#pragma once
#include "awm_kernels.cuh"
#include "awm_tc.cuh"
#include <cuda_fp16.h>

namespace awm {

constexpr int kTcTile = 128;                 // frames per tile = UMMA M
constexpr int kTcK = 96;                     // 81 bands padded to a multiple of the UMMA K (16)
constexpr uint32_t kTcASplit = kTcTile * kTcK * 2;        // bytes of one fp16 term of the A tile (24 KB)
constexpr uint32_t kTcABytes = 2 * kTcASplit;             // hi + lo
constexpr int kTcEpiWarps = 4;
// CHUNK_ENT sync entries per B chunk -> UMMA N = 2 CHUNK_ENT (U and D column of every entry), chunk of N x 96 fp16.
// 128 entries (N = 256, 48 KB) with eight FFT warps; 48 entries (N = 96, 18 KB) leave room for twelve FFT warps AND two A buffers.
__host__ __device__ constexpr uint32_t tc_b_bytes (int chunk_ent) { return uint32_t (2 * chunk_ent) * kTcK * 2; }
__host__ __device__ constexpr int tc_tmem_columns (int chunk_ent) { return 4 * chunk_ent <= 32 ? 32 : 4 * chunk_ent <= 64 ? 64 : 4 * chunk_ent <= 128 ? 128 : 4 * chunk_ent <= 256 ? 256 : 512; }

template<int FFT_WARPS, int A_BUFS, int CHUNK_ENT> constexpr size_t
tc_smem_bytes() { return fft_smem_bytes (FFT_WARPS) + size_t (A_BUFS) * kTcABytes + tc_b_bytes (CHUNK_ENT) + 256; }

// host side: the 0/1 masks of all entries in operand layout, chunk after chunk ([ceil (n_ent / chunk_ent)][tc_b_bytes (chunk_ent)])
inline void
tc_build_masks (const awm_sync_entry *ent, int n_ent, int chunk_ent, std::vector<unsigned char>& out)
{
  const int n_chunks = (n_ent + chunk_ent - 1) / chunk_ent;
  const size_t b_bytes = tc_b_bytes (chunk_ent);
  out.assign (size_t (n_chunks) * b_bytes, 0);
  const uint16_t one = 0x3c00;               // 1.0 in fp16
  for (int e = 0; e < n_ent; e++)
    {
      unsigned char *chunk = out.data() + size_t (e / chunk_ent) * b_bytes;
      const int col = 2 * (e % chunk_ent);
      for (int i = 0; i < kUD; i++)
        {
          memcpy (chunk + tc::operand_offset (2 * chunk_ent, col, ent[e].up[i]), &one, 2);
          memcpy (chunk + tc::operand_offset (2 * chunk_ent, col + 1, ent[e].down[i]), &one, 2);
        }
    }
}

template<int FFT_WARPS, int A_BUFS, int CHUNK_ENT> __global__ void __launch_bounds__ ((FFT_WARPS + kTcEpiWarps + 1) * 32, 1)
k_stft_mags_tc (const float *__restrict__ pcm, long long n_frames, int C, int n_out, int ld,
                const unsigned char *__restrict__ masks /* [n_chunks][tc_b_bytes (CHUNK_ENT)] */, int n_ent, int n_chunks,
                float2 *__restrict__ mags /* [4][n_ent][ld] */, unsigned char *__restrict__ have,
                long long wav_first, long long wav_last, const float2 *g_tw, const float *g_win, int tma_ok /* stereo, pcm 16-byte aligned */)
{
  using namespace tc;
  constexpr int kTcChunkEnt = CHUNK_ENT, kTcN = 2 * CHUNK_ENT;
  constexpr uint32_t kTcBBytes = tc_b_bytes (CHUNK_ENT);
  constexpr int kTmemCols = tc_tmem_columns (CHUNK_ENT);
  extern __shared__ __align__ (16) unsigned char smem[];
  FftSmem s = fft_smem_setup (smem, g_tw, g_win, FFT_WARPS);
  unsigned char *abuf = reinterpret_cast<unsigned char *> (s.extra);
  unsigned char *bbuf = abuf + size_t (A_BUFS) * kTcABytes;
  uint64_t *bars = reinterpret_cast<uint64_t *> (bbuf + kTcBBytes);
  uint64_t *a_full = bars, *a_empty = bars + 2, *b_full = bars + 4, *b_free = bars + 5, *tmem_full = bars + 6, *tmem_empty = bars + 8;
  uint64_t *pcm_bars = bars + 10;                                  // one per FFT warp: its next frame has landed in its transpose buffer
  uint32_t *tmem_slot = reinterpret_cast<uint32_t *> (pcm_bars + FFT_WARPS);
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  constexpr int kMmaWarp = FFT_WARPS + kTcEpiWarps;

  if (threadIdx.x == 0)
    {
      for (int i = 0; i < 2; i++)
        {
          mbar_init (&a_full[i], FFT_WARPS);
          mbar_init (&a_empty[i], 1);
          mbar_init (&tmem_full[i], 1);
          mbar_init (&tmem_empty[i], kTcEpiWarps);
        }
      mbar_init (b_full, 1);
      mbar_init (b_free, 1);
      for (int i = 0; i < FFT_WARPS; i++)
        mbar_init (&pcm_bars[i], 1);
      fence_mbar_init();
    }
  if (w == kMmaWarp)
    tmem_alloc (tmem_slot, kTmemCols);
  // band columns 81 .. 95 of A are never written again and must be finite: clear everything once
  for (uint32_t i = threadIdx.x; i < A_BUFS * kTcABytes / 16; i += blockDim.x)
    reinterpret_cast<uint4 *> (abuf)[i] = make_uint4 (0, 0, 0, 0);
  fence_proxy_async();
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const int n_tiles = 4 * ((n_out + kTcTile - 1) / kTcTile);

  if (w < FFT_WARPS)
    {
      // ===================================================================================== FFT warps
      // The PCM of a frame reaches the warp through the bulk-copy engine: while the second butterfly pass of frame i runs, the
      // 8 KB of frame i + 1 (1024 stereo sample-frames, contiguous and 16-byte aligned in the interleaved stream) land in the
      // warp's transpose buffer, which is idle from that point on; the next iteration finds them in shared memory (mbarrier
      // complete_tx) instead of waiting ~1 us for 32 global loads per lane.  Frames the copy cannot serve -- mono / multichannel
      // audio, the ragged end of the stream, an unaligned caller buffer -- take the global-load path of frame_db_sum.
      uint64_t *pcm_bar = pcm_bars + w;
      uint32_t pcm_phase = 0;
      struct Frame { int t, r; };
      auto frame_start = [&] (Frame fr) { return (long long) (fr.t & 3) * 256 + (long long) ((fr.t >> 2) * kTcTile + fr.r) * kFrame; };
      auto exists = [&] (Frame fr) { return fr.t < n_tiles; };
      auto wanted = [&] (Frame fr)          // sync_fft computes this frame: inside the output range and not in leading / trailing digital silence
        {
          const long long start = frame_start (fr);
          const long long f_first = start * C, f_last = (start + kFrame) * C;
          return (fr.t >> 2) * kTcTile + fr.r < n_out && !(f_last < wav_first || f_first > wav_last);
        };
      auto by_tma = [&] (Frame fr) { return tma_ok && exists (fr) && wanted (fr) && frame_start (fr) + kFrame <= n_frames; };
      auto next_of = [&] (Frame fr)
        {
          fr.r += FFT_WARPS;
          if (fr.r >= kTcTile)
            {
              fr.r = w;
              fr.t += gridDim.x;
            }
          return fr;
        };
      auto prefetch = [&] (Frame fr)        // caller: after __syncwarp, every lane is done with the transpose buffer
        {
          if (lane == 0)
            {
              fence_proxy_async();          // the lanes' generic-proxy accesses to xbuf are ordered before the engine's writes
              mbar_arrive_expect_tx (pcm_bar, kFrame * 2 * sizeof (float));
              bulk_load (s.xbuf, pcm + frame_start (fr) * 2, kFrame * 2 * sizeof (float), pcm_bar);
            }
        };
      Frame cur { int (blockIdx.x), w };
      if (by_tma (cur))
        prefetch (cur);
      int it = 0;
      for (; exists (cur); it++)
        {
          const int shift_idx = cur.t & 3, f0 = (cur.t >> 2) * kTcTile;
          const int a = it % A_BUFS, use = it / A_BUFS;
          mbar_wait_relaxed (&a_empty[a], (use & 1) ^ 1);         // the MMAs that read this buffer last time are done
          unsigned char *A = abuf + size_t (a) * kTcABytes;
          const int t_now = cur.t;
          for (; cur.t == t_now; )
            {
              const int r = cur.r, f = f0 + r;
              const Frame nxt = next_of (cur);
              const bool ok = wanted (cur), nxt_tma = by_tma (nxt);
              float acc[4] = { 0.f, 0.f, 0.f, 0.f };
              if (by_tma (cur))
                {
                  float re[32], im[32];
                  mbar_wait (pcm_bar, pcm_phase);
                  pcm_phase ^= 1;
                  const float2 *xp = reinterpret_cast<const float2 *> (s.xbuf) + lane;
#pragma unroll
                  for (int j = 0; j < 32; j++)
                    {
                      const float2 v = xp[32 * j];
                      const float wn = s.win[32 * j + lane];
                      re[j] = __fmul_rn (v.x, wn);
                      im[j] = __fmul_rn (v.y, wn);
                    }
                  __syncwarp();                                   // all lanes hold their samples before the transposes reuse the buffer
                  const unsigned zero = pair_zero_mask (re, im);
                  fft1024_warp (re, im, s.tw, s.xbuf, lane, [&] { if (nxt_tma) prefetch (nxt); });
                  // dB with MUFU.LG2 (__log2f): its error (~2e-7 relative) is two orders below the 2^-16 absolute resolution the
                  // value is about to be stored with (fp16 hi + lo), and saves ~170 of the ~2000 instructions of a frame
                  auto db = [] (float re_, float im_) { const float a2 = __fmaf_rn (re_, re_, __fmul_rn (im_, im_)); return a2 > 0.0f ? __log2f (a2) * 3.01029995663981f : -96.f; };
                  float ar, ai, br, bi;
                  unpack_pair<0> (re, im, lane, ar, ai, br, bi, zero);
                  acc[0] = db (ar, ai) + db (br, bi);
                  unpack_pair<1> (re, im, lane, ar, ai, br, bi, zero);
                  acc[1] = db (ar, ai) + db (br, bi);
                  unpack_pair<2> (re, im, lane, ar, ai, br, bi, zero);
                  acc[2] = db (ar, ai) + db (br, bi);
                  unpack_pair<3> (re, im, lane, ar, ai, br, bi, zero);
                  acc[3] = db (ar, ai) + db (br, bi);
                }
              else
                {
                  if (ok)
                    frame_db_sum (pcm, n_frames, C, frame_start (cur), s, lane, acc);
                  __syncwarp();
                  if (nxt_tma)
                    prefetch (nxt);
                }
#pragma unroll
              for (int k2 = 0; k2 < 4; k2++)
                {
                  const int band = lane + 32 * k2 - kMinBand;
                  if (band >= 0 && band < kBands)
                    {
                      const __half hi = __float2half_rn (acc[k2]);
                      const __half lo = __float2half_rn (acc[k2] - __half2float (hi));
                      const uint32_t o = operand_offset (kTcTile, r, band);
                      *reinterpret_cast<__half *> (A + o) = hi;
                      *reinterpret_cast<__half *> (A + kTcASplit + o) = lo;
                    }
                }
              if (lane == 0 && f < n_out)
                have[(size_t) shift_idx * ld + f] = ok ? 1 : 0;
              cur = nxt;
            }
          fence_proxy_async();                                    // st.shared above -> visible to tcgen05.mma (async proxy)
          __syncwarp();
          if (lane == 0)
            mbar_arrive (&a_full[a]);
        }
    }
  else if (w < kMmaWarp)
    {
      // ===================================================================================== epilogue warps
      const int q = w & 3;                                        // a warp reaches the TMEM lanes of its quadrant only: 32 q .. 32 q + 31 (the four epilogue warps are consecutive, so every quadrant is served)
      int g = 0;
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x)
        {
          const int shift_idx = t & 3, f0 = (t >> 2) * kTcTile;
          const int f = f0 + q * 32 + lane;                       // frame of this thread's TMEM lane; f < ld always (ld multiple of 128)
          for (int c = 0; c < n_chunks; c++, g++)
            {
              const int tb = g & 1;
              mbar_wait_relaxed (&tmem_full[tb], (g >> 1) & 1);
              tc_fence_after_sync();
              const uint32_t taddr = tmem + (uint32_t (q * 32) << 16) + uint32_t (tb * kTcN);
#pragma unroll 1
              for (int c0 = 0; c0 < kTcN; c0 += 32)
                {
                  uint32_t r[32];
                  tmem_ld_32x32 (taddr + c0, r);
                  tmem_ld_wait();
                  const int e0 = c * kTcChunkEnt + c0 / 2;
#pragma unroll
                  for (int p = 0; p < 16; p++)
                    if (e0 + p < n_ent)                           // warp uniform
                      mags[((size_t) shift_idx * n_ent + e0 + p) * ld + f] = make_float2 (__uint_as_float (r[2 * p]), __uint_as_float (r[2 * p + 1]));
                }
              tc_fence_before_sync();
              __syncwarp();
              if (lane == 0)
                mbar_arrive (&tmem_empty[tb]);
            }
        }
    }
  else if (lane == 0)
    {
      // ===================================================================================== TMA + MMA issue (one thread)
      constexpr uint32_t idesc = idesc_f16_f32 (kTcTile, kTcN);
      const uint32_t b_addr = smem_u32 (bbuf);
      int it = 0, g = 0;
      for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, it++)
        {
          const int a = it % A_BUFS, use = it / A_BUFS;
          const uint32_t a_addr = smem_u32 (abuf + size_t (a) * kTcABytes);
          for (int c = 0; c < n_chunks; c++, g++)
            {
              if (g > 0)
                mbar_wait_relaxed (b_free, (g - 1) & 1);                      // the MMAs of the previous chunk have read the B buffer
              mbar_arrive_expect_tx (b_full, kTcBBytes);
              bulk_load (bbuf, masks + size_t (c) * kTcBBytes, kTcBBytes, b_full);
              if (c == 0)
                mbar_wait_relaxed (&a_full[a], use & 1);                // all FFT warps have delivered their rows of the tile
              mbar_wait_relaxed (b_full, g & 1);
              const int tb = g & 1;
              mbar_wait_relaxed (&tmem_empty[tb], ((g >> 1) & 1) ^ 1);    // the epilogue has drained this accumulator
              tc_fence_after_sync();
#pragma unroll
              for (int sp = 0; sp < 2; sp++)
#pragma unroll
                for (int j = 0; j < kTcK / 16; j++)
                  mma_f16 (tmem + uint32_t (tb * kTcN),
                           smem_desc_kmajor (a_addr + sp * kTcASplit + j * 2 * (kTcTile * 16), kTcTile * 16, 128),
                           smem_desc_kmajor (b_addr + j * 2 * (kTcN * 16), kTcN * 16, 128), idesc, (sp | j) != 0);
              mma_commit (b_free);
              mma_commit (&tmem_full[tb]);
            }
          mma_commit (&a_empty[a]);
        }
    }
  tc_fence_before_sync();
  __syncthreads();
  if (w == kMmaWarp)
    {
      tc_fence_after_sync();
      tmem_dealloc (tmem, kTmemCols);
    }
}

} // namespace awm
