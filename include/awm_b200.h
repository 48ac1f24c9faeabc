/* awm_b200.h -- C ABI of the B200-native spectral watermark hot path.
 *
 * The reference (swesterfeld/audiowmark) has no FFI: its hot path is reached through
 * C++ classes and three free functions.  This header is the boundary a maintainer would
 * bind instead; every entry point names the reference interface it replaces
 * (paths relative to the reference tree).  Plain pointers and sizes only.
 *
 * Conventions
 *  - every function returns 0 on success, nonzero on error; awm_last_error (ctx) gives the text
 *  - a context owns one CUDA device + stream; single-owner, calls are stream ordered
 *  - PCM is interleaved fp32 in [-1,1) (what AudioInputStream::read_frames delivers,
 *    src/audiostream.hh:41-52); pointers may be host or device memory
 *  - "frame" in argument names is one PCM sample-frame (one sample per channel)
 *  - there is NO CPU fallback: without a usable CUDA device awm_create fails
 */
#ifndef AWM_B200_H
#define AWM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct awm_ctx awm_ctx;

#define AWM_FRAME_SIZE   1024   /* Params::frame_size      src/wmcommon.hh:36 */
#define AWM_MIN_BAND     20     /* Params::min_band        src/wmcommon.hh:40 */
#define AWM_MAX_BAND     100    /* Params::max_band        src/wmcommon.hh:39 */
#define AWM_N_BANDS      81
#define AWM_BANDS_PER_FRAME 30  /* Params::bands_per_frame src/wmcommon.hh:38 */
#define AWM_VITERBI_ORDER 15    /* src/convcode.cc:49 */

enum { AWM_MODE_BLOCK = 0, AWM_MODE_CLIP = 1 };           /* SyncFinder::Mode, src/syncfinder.hh:71 */
enum { AWM_BLOCK_A = 0, AWM_BLOCK_B = 1, AWM_BLOCK_AB = 2 }; /* ConvBlockType, src/convcode.hh:24 */

/* One sync frame: SyncFinder::FrameBit (src/syncfinder.hh:78-83); band indices are bin - AWM_MIN_BAND */
typedef struct {
  uint16_t frame;
  uint8_t  up[AWM_BANDS_PER_FRAME];
  uint8_t  down[AWM_BANDS_PER_FRAME];
} awm_sync_entry;

/* One mix entry: MixEntry (src/wmcommon.hh:149-154); up/down are FFT bin numbers */
typedef struct {
  uint16_t frame;
  uint8_t  up;
  uint8_t  down;
} awm_mix_entry;

/* SyncFinder::SearchScore (src/syncfinder.hh:89-98) */
typedef struct {
  uint64_t index;
  double   raw_quality;
  double   local_mean;
} awm_search_score;

/* ---- lifetime ------------------------------------------------------------------------- */
int         awm_create (int device, awm_ctx **out);
void        awm_destroy (awm_ctx *ctx);
const char *awm_last_error (const awm_ctx *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t    awm_launch_count (const awm_ctx *ctx);
/* CUDA stream (cudaStream_t) the context launches on, for event timing by the caller */
void       *awm_stream (awm_ctx *ctx);
int         awm_synchronize (awm_ctx *ctx);
/* measurement aid: when enabled every kernel launch is bracketed by CUDA events on the context stream;
 * awm_profile_report synchronises, writes {"kernel": {"launches": n, "ms": total}, ...} as JSON and resets */
/* page-locked host memory for buffers that cross PCIe (PCM, score lists); plain malloc'ed memory works too, only slower */
void       *awm_host_alloc (size_t bytes);
void        awm_host_free (void *p);
int         awm_profile_enable (awm_ctx *ctx, int on);
int         awm_profile_report (awm_ctx *ctx, char *json_out, size_t json_cap);

/* ---- FFTProcessor (src/fft.hh:25-44, src/fft.cc:82-118) ------------------------------------
 * batched r2c / unnormalised c2r, n must be 1024.  in/out layouts as FFTW:
 *   r2c: in [count][1024] real  -> out [count][1026] (513 complex, re/im interleaved)
 *   c2r: in [count][1026]       -> out [count][1024] (sum over the Hermitian extension, not divided by n)
 */
int awm_fft_r2c (awm_ctx *ctx, const float *in, float *out, size_t count, int n);
int awm_fft_c2r (awm_ctx *ctx, const float *in, float *out, size_t count, int n);

/* ---- key / payload derived tables (built on the host, the AES key never reaches the GPU) ----
 * embed : FrameMod table of init_frame_mod_vec (src/wmadd.cc:148-162): uint8 [2 (A,B)][frames_per_block][101],
 *         0 keep / 1 up / 2 down
 * sync  : SyncFinder::get_sync_bits (src/syncfinder.cc:30-77) flattened bit-major; bit b owns
 *         entries bit_offsets[b] .. bit_offsets[b+1]-1, entries sorted by frame inside a bit
 * mix   : gen_mix_entries (src/wmcommon.cc:179-202) and the bit order permutation of
 *         randomize_bit_order (src/wmcommon.hh:165-185): out[bit_order[i]] = in[i] on decode
 * key_slot selects one of AWM_MAX_KEYS table sets (audiowmark get accepts several --key options).
 */
#define AWM_MAX_KEYS 16
int awm_set_embed_tables (awm_ctx *ctx, const uint8_t *frame_mod_ab, int frames_per_block);
int awm_set_sync_tables (awm_ctx *ctx, int key_slot, int mode, const awm_sync_entry *entries, int n_entries,
                         const int *bit_offsets, int n_bits);
int awm_set_mix_tables (awm_ctx *ctx, int key_slot, const awm_mix_entry *entries, int n_entries,
                        const uint16_t *bit_order, int n_coded_bits, int frames_per_bit, int frames_per_block);

/* ---- PCM residency (WavData::samples, src/wavdata.hh:27-74) ---------------------------------
 * Binds the audio the following sync / decode calls work on.  A host pointer is copied to a
 * context-owned device buffer (pinned or pageable, async on the context stream); a device
 * pointer is used in place and must stay valid until the next bind.
 * pad_start/pad_end: that many zero sample-frames are logically prepended / appended
 * (ClipDecoder::run_block zero padding, src/wmget.cc:823-866) without the caller materialising them.
 */
int awm_pcm_bind (awm_ctx *ctx, const float *pcm, size_t n_frames, int channels, size_t pad_start, size_t pad_end);
/* optional: start copying a HOST buffer that will be bound next (the following chunk of a long file) on a separate
 * stream while the kernels of the current chunk run; a later awm_pcm_bind with the same pointer / size / channels and
 * no padding picks the copy up instead of transferring again.  Two prefetches may be outstanding.  A span that starts inside
 * the still unbound span prefetched just before it, in the same host buffer (the overlapping chunks of WavChunkLoader,
 * src/wavchunkloader.cc:54-163), takes its head from that device copy and only transfers the rest; the host memory of an unbound
 * prefetch must not change meanwhile.  Spans in different host buffers: awm_pcm_prefetch_wav marks the overlap explicitly. */
int awm_pcm_prefetch (awm_ctx *ctx, const float *pcm, size_t n_frames, int channels);

/* 16 bit PCM variants: the buffers hold interleaved int16 (what a 16 bit WAV file holds); conversion to / from the float
 * pipeline happens on the device with the reference's rules -- reading: sample * 2^-15 (src/sfinputstream.cc:189-210),
 * writing: float_to_int_clip<32> (src/rawconverter.hh:34-50), 16 most significant bits kept (src/sfoutputstream.cc:148-155) --
 * so results are identical to converting on the host, at half the PCIe traffic. */
int awm_pcm_bind_s16 (awm_ctx *ctx, const int16_t *pcm, size_t n_frames, int channels, size_t pad_start, size_t pad_end);
int awm_pcm_prefetch_s16 (awm_ctx *ctx, const int16_t *pcm, size_t n_frames, int channels);
/* Any sample format a WAV file of `get` can store, decoded on the device (the _s16 entry points above are the 16 bit case):
 *   bits 8 (unsigned, as WAV stores 8 bit), 16, 24, 32 with is_float = 0: little-endian integers, left justified to 32 bits and
 *   multiplied by 2^-31 in float; bits 32, 64 with is_float = 1: little-endian IEEE floats, doubles rounded to float.
 * The rules are RawConverter::from_raw's (src/rawconverter.cc), so the bound floats are bit-identical to a host conversion
 * (NaN, Inf, denormals and values beyond +-1 included) while only the stored bytes cross PCIe.  `bytes` may start at any address.
 * awm_pcm_bind_wav: as awm_pcm_bind.
 * awm_pcm_prefetch_wav: as awm_pcm_prefetch, but the caller marks the overlap with the previous span itself, so that consecutive
 *   spans may sit in different host buffers (WavChunkLoader's chunks read into two buffers in turn, src/wavchunkloader.cc:54-163):
 *   the first head_frames frames of the span are the last head_frames frames of the span prefetched just before it (same format
 *   and channels; bound since or not) and are copied on the device; `bytes` holds only the n_frames - head_frames frames after
 *   them, and only those cross PCIe.  Bind the span with the same `bytes` pointer and the full n_frames.  The host bytes must not
 *   change until the span is bound. */
typedef struct {
  int bits;                     /* 8, 16, 24, 32 or 64 */
  int is_float;                 /* 0: integer PCM, 1: IEEE float */
} awm_wav_format;
int awm_pcm_bind_wav (awm_ctx *ctx, const void *bytes, awm_wav_format format, size_t n_frames, int channels, size_t pad_start, size_t pad_end);
int awm_pcm_prefetch_wav (awm_ctx *ctx, const void *bytes, awm_wav_format format, size_t n_frames, int channels, size_t head_frames);
/* A long HOST stream (float or 16 bit PCM) on its way to the device piece by piece, for callers that work on parts of it while the
 * rest is still crossing PCIe (the sharded get: a rank searches its first chunk slice while its later slices arrive; replaces the
 * read-ahead of WavChunkLoader, src/wavchunkloader.cc:54-163).  awm_pcm_stage starts the copies on a copy stream and returns the
 * device address of the float copy at once; awm_pcm_stage_wait (n) orders everything issued on the context stream afterwards
 * behind the arrival of the first n sample-frames.  Bind parts with awm_pcm_bind (device pointer + offset). */
int awm_pcm_stage (awm_ctx *ctx, const void *pcm, int is_s16, size_t n_frames, int channels, size_t piece_frames, const float **device_out);
int awm_pcm_stage_wait (awm_ctx *ctx, size_t n_frames);
/* device copy (float) of the bound PCM incl. padding; NULL if nothing is bound */
const float *awm_pcm_device (awm_ctx *ctx, size_t *n_frames, int *channels);

/* ---- embed: add_stream_watermark main loop (src/wmadd.cc:520-589) = FFTAnalyzer::run_fft
 * (src/wmcommon.cc:91-121) + apply_frame_mod (src/wmadd.cc:61-84) + WatermarkSynth::run
 * (src/wmadd.cc:215-250) + mix + Limiter::process (src/limiter.cc:45-124), for a whole buffer
 * at 44.1 kHz.  in/out: [n_frames][channels]; first_frame_number = index of the first 1024-frame
 * of this buffer in the stream (0 unless the caller shards; WatermarkGen starts its table row
 * at 2*frames_per_block - frames_pad_start, src/wmadd.cc:295; limiter blocks are counted from the stream start
 * as well, so a shard that brings a halo of one frame + two limiter blocks on each side reproduces the
 * unsharded result exactly in its interior).  limiter_block = sample_rate *
 * 1000 / 1000 frames (src/limiter.cc:33-37); limiter_block = 0 disables the limiter
 * (--test-no-limiter).  snr_power (optional, 2 doubles) receives sum(delta^2), sum(orig^2)
 * as --snr accumulates them (src/wmadd.cc:553-563).
 */
int awm_embed (awm_ctx *ctx, const float *in, float *out, size_t n_frames, int channels,
               uint64_t first_frame_number, int frames_pad_start, double water_delta,
               int limiter_block, float limiter_ceiling, double *snr_power);
/* awm_embed for one WINDOW of a longer stream (streaming `add` with bounded memory, add_stream_watermark's loop src/wmadd.cc:520-589
 * taken window by window): the buffer holds the window plus its halo, first_frame_number places it in the stream; only positions
 * [snr_first, snr_last) of the buffer (the part the caller keeps) enter the --snr sums.  Everything else as awm_embed. */
int awm_embed_window (awm_ctx *ctx, const float *in, float *out, size_t n_frames, int channels,
                      uint64_t first_frame_number, int frames_pad_start, double water_delta,
                      int limiter_block, float limiter_ceiling, uint64_t snr_first, uint64_t snr_last, double *snr_power);
/* the same for 16 bit PCM in and out (see awm_pcm_bind_s16): what `audiowmark add in16.wav out16.wav` computes between the files */
int awm_embed_s16 (awm_ctx *ctx, const int16_t *in, int16_t *out, size_t n_frames, int channels,
                   uint64_t first_frame_number, int frames_pad_start, double water_delta,
                   int limiter_block, float limiter_ceiling, double *snr_power);

/* ---- sync search on the bound PCM --------------------------------------------------------
 * awm_sync_approx = SyncFinder::search_approx (src/syncfinder.cc:171-256): for the four
 * 256-sample shifts the channel-summed dB spectrogram (sync_fft, :560-605), sync_decode (:116-153)
 * for every start frame, and the local mean (:234-254).  scores_out (device->host) receives
 * *n_scores entries sorted by index.  wav_first/wav_last: non-silent value range
 * [first,last) as scan_silence computes it (:155-169) in interleaved-value units of the padded
 * signal; pass 0 / n_values for BLOCK mode.
 * Passing scores_out = NULL runs the search, keeps the scores on the device (for awm_sync_peaks) and returns the count.
 */
int awm_sync_approx (awm_ctx *ctx, int key_slot, int mode, uint64_t wav_first, uint64_t wav_last,
                     double water_delta, awm_search_score *scores_out, size_t max_scores, size_t *n_scores);

/* awm_sync_peaks = sync_select_local_maxima (src/syncfinder.cc:258-281) on the score list of the last
 * awm_sync_approx call (kept on the device), restricted to peaks with |raw_quality - local_mean| > min_abs_quality:
 * only those can pass the threshold / n-best selection that follows, so the host never has to look at the
 * several hundred thousand scores of a 30 minute chunk.  out: sorted by index; *n = number found (may exceed max,
 * then only max entries were written and the caller should raise min_abs_quality or use awm_sync_approx's full list).
 */
int awm_sync_peaks (awm_ctx *ctx, double min_abs_quality, awm_search_score *out, size_t max, size_t *n);

/* awm_sync_refine = SyncFinder::search_refine (src/syncfinder.cc:393-458): for each candidate the
 * fine offsets max(index-256,0) .. index+256 step 8 are scored with fresh FFTs of the wanted
 * sync frames; in/out: index, raw_quality are replaced by the best offset (strict '>' on
 * |q - local_mean|, earlier offset wins ties), local_mean is kept.
 */
int awm_sync_refine (awm_ctx *ctx, int key_slot, int mode, uint64_t wav_first, uint64_t wav_last,
                     double water_delta, awm_search_score *scores, size_t n_scores);

/* measurement aid for the parity tests: the sync_decode quality of each of the 65 fine offsets search_refine looks at
 * (src/syncfinder.cc:428-434), as the sliding-DFT kernel ranks them (exact = 0) or from fresh transforms in the reference's
 * summation order (exact = 1).  quality_out / valid_out: [n_scores][65]; offsets the reference gets no result for
 * (sync_fft returns nothing past the end of the signal) have valid 0.  awm_sync_refine re-scores every offset whose sliding
 * quality is within 1e-3 of the best exactly, so its result is that of the exact kernel as long as the two differ by < 5e-4. */
int awm_sync_refine_offsets (awm_ctx *ctx, int key_slot, int mode, uint64_t wav_first, uint64_t wav_last, double water_delta,
                             const awm_search_score *scores, size_t n_scores, int exact, double *quality_out, unsigned char *valid_out);

/* ---- block decode: FFTAnalyzer::fft_range (src/wmcommon.cc:123-141) + mix_decode
 * (src/wmget.cc:67-108) + randomize_bit_order(decode) for blocks starting at indices[i]
 * (sample-frames of the padded signal).  raw_bits_out: [n_blocks][n_coded_bits] floats;
 * valid_out[i] = 0 when the block would read past the end (fft_range returns empty).
 */
int awm_decode_blocks (awm_ctx *ctx, int key_slot, const uint64_t *indices, size_t n_blocks,
                       float *raw_bits_out, int *valid_out);

/* ---- Viterbi: normalize_soft_bits (src/wmget.cc:40-65) + conv_decode_soft (src/convcode.cc:128-213)
 * for n_jobs independent code words in one launch.  block_types[j] in AWM_BLOCK_*: A / B words carry
 * 6 * (n_msg_bits + 15) soft bits, AB words 12 * (n_msg_bits + 15); raw_bits holds the jobs back to back
 * (un-normalised soft bits as mix_decode delivers them); hard != 0 => --hard.
 * bits_out: [n_jobs][n_msg_bits] bytes (0/1), error_out[j] = final path metric / coded bits.
 */
int awm_viterbi (awm_ctx *ctx, const float *raw_bits, size_t n_jobs, int n_msg_bits, const int *block_types,
                 int hard, uint8_t *bits_out, float *error_out);

/* ---- resampler: process_resampler / resample / resample_ratio_truncate (src/resample.cc:27-131) -------------
 * The reference delegates to zita-resampler (third party, not part of its tree); this library defines the filter itself:
 *   out[n] = sum_i in[i] g (i - n / ratio),   g (d) = fc sinc (fc d) w (d / h),   fc = min (1, ratio),   h = ceil (hlen / fc),
 *   w = 0.384 + 0.5 cos (pi x) + 0.116 cos (2 pi x) on [-1, 1];  256 phases, linear interpolation between phase rows,
 *   float accumulation in tap order; in is zero outside [0, n_in), outputs whose taps would pass h frames beyond the
 *   input are 0 (where a streaming resampler fed h - 1 frames of pre-roll and h of post-roll stops).
 * in/out: interleaved, host or device.  hlen = 16 everywhere in the reference.
 */
int awm_resample (awm_ctx *ctx, const float *in, size_t n_in, int channels, double ratio, int hlen, float *out, size_t n_out);

/* ---- embed for inputs that are not at the watermark rate: WatermarkResampler::run (src/wmadd.cc:353-430) inside the
 * add loop (:520-589).  The input is resampled to mark_sample_rate, the watermark signal alone is generated there
 * (WatermarkGen::run), resampled back and added to the untouched input; the limiter runs at the input rate
 * (limiter_block = sample_rate * ms / 1000).  n_emit >= n_frames = frames the reference loop pushes through the mixer
 * before it stops (zero frames are fed after EOF until resamplers and limiter have delivered everything): they enter the
 * --snr sums and the limiter's block peaks.  in/out: [n_frames][channels], host or device.
 */
int awm_embed_resampled (awm_ctx *ctx, const float *in, float *out, size_t n_frames, int channels, int sample_rate, int mark_sample_rate,
                         size_t n_emit, int frames_pad_start, double water_delta, int limiter_block, float limiter_ceiling, double *snr_power);

/* resample_ratio (wav_data, speed, ...) of decode() (src/wmget.cc:916) without leaving the device: the bound PCM is
 * resampled by `ratio` into a context-owned buffer of n_out frames, which becomes the bound PCM; awm_pcm_pop restores
 * the previous binding (the original chunk is not copied again).  One level only; awm_pcm_bind drops a pushed binding. */
int awm_pcm_push_resampled (awm_ctx *ctx, double ratio, int hlen, size_t n_out);
int awm_pcm_pop (awm_ctx *ctx);
/* stream ordered copy device (or host) -> host for callers that keep their PCM in device memory but need a few values on
 * the host (clip selection of detect_speed hashes a sparse subset of the samples, src/wmspeed.cc:533-552) */
int awm_copy_to_host (awm_ctx *ctx, void *dst, const void *src, size_t bytes);
/* dst_host[k] = src[indices[k]] for a device resident src (the sample subset detect_speed hashes) */
int awm_gather (awm_ctx *ctx, const float *src, const uint64_t *indices, size_t n, float *dst_host);
/* 1 if p points to CUDA device / managed memory (such pointers are used in place by the PCM entry points), else 0 */
int awm_is_device_pointer (const void *p);

/* ---- speed detection scan: SpeedSync::prepare_mags + SpeedSync::compare (src/wmspeed.cc:203-375) ------------------
 * clip = the audio SpeedSearch::get_jobs cut out (get_speed_clip, :33-52).  For every centre speed the clip is
 * truncated to seconds / centre, resampled by centre / 2, turned into the MagMatrix (512-point spectra, hop 128), and
 * scored for n_relative relative speeds (relative_speeds[c * n_relative + r] = pow (step, p) * speed / centre, :173).
 * quality_out[c * n_relative + r] = Score::quality of that compare() call (0 if no offset had data).
 * Uses the BLOCK mode sync table of key_slot (awm_set_sync_tables) and frames_per_block of awm_set_mix_tables.
 */
int awm_speed_scan (awm_ctx *ctx, int key_slot, const float *clip, size_t clip_frames, int channels, int sample_rate,
                    double seconds, const double *centers, int n_centers, const double *relative_speeds, int n_relative,
                    double water_delta, double *quality_out);

/* ---- multi-GPU exchange for the sharded `get` (one process per GPU) ------------------------------------------------------
 * The reference has no counterpart: its thread pool shares one address space.  Here the ranks of a job exchange the small
 * per-chunk lists of the search (peaks, refined scores + soft bits, decoded words) with ncclAllGather on the context stream;
 * no PCM ever crosses NVLink.  awm_dist_unique_id: rank 0 creates the NCCL id, the launcher hands it to every rank (bench.py
 * broadcasts it with torch.distributed); awm_dist_init joins the communicator; awm_dist_allgather: every rank contributes
 * send_bytes (<= slot_bytes - 8) and receives rank r's bytes at recv + r * slot_bytes, its length in recv_bytes[r].  Returns 2
 * when some rank's payload did not fit (recv_bytes then holds all lengths: repeat with a larger slot; every rank sees the same).
 * Without awm_dist_init the "world" is this process alone and the call degenerates to a copy. */
int awm_dist_unique_id (unsigned char id_out[128]);
int awm_dist_init (awm_ctx *ctx, int rank, int world, const unsigned char id[128]);
int awm_dist_world (const awm_ctx *ctx, int *rank, int *world);
int awm_dist_allgather (awm_ctx *ctx, const void *send, size_t send_bytes, size_t slot_bytes, void *recv, size_t *recv_bytes);

#ifdef __cplusplus
}
#endif
#endif /* AWM_B200_H */
