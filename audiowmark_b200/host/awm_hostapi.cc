// awm_hostapi.cc -- plain C entry points over the host-side C++ (tables, add, get) so that the parity
// tests and bench.py can drive exactly what the CLI runs.  Table functions are pure host code (no GPU).
#include "awm_results.hh"
#include "awm_balanced.hh"
#include "awm_speed.hh"
#include "awm_engine.hh"
#include "awm_tables.hh"
#include "awm_util.hh"

#include <algorithm>
#include <math.h>
#include <memory>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static Key
make_key (const unsigned char *key16, const char *name)
{
  Key k;
  k.set_key (key16, name ? name : "");
  return k;
}

std::vector<unsigned char> block_jobs_blob (const Key& key, const std::vector<SyncFinder::Score>& sync_scores, const std::vector<std::vector<float>>& raw,
                                            const std::vector<int>& valid, int sample_rate, int *n_jobs);

extern "C" {

void
awmh_set_params (double water_delta, int frames_per_bit, int mix, int hard, double sync_threshold2, int n_best,
                 double chunk_size_min, int test_no_limiter, int test_no_sync, int gpu_device, int quiet)
{
  Params::water_delta = water_delta;
  Params::frames_per_bit = frames_per_bit;
  Params::mix = mix != 0;
  Params::hard = hard != 0;
  Params::sync_threshold2 = sync_threshold2;
  Params::get_n_best = n_best;
  Params::get_chunk_size = chunk_size_min;
  Params::test_no_limiter = test_no_limiter != 0;
  Params::test_no_sync = test_no_sync != 0;
  Params::gpu_device = gpu_device;
  set_log_level (quiet ? Log::WARNING : Log::INFO);
}

/* --short <bits> (src/audiowmark.cc:665-674); bits = 0 returns to the 128 bit payload.  returns the block code length or -1 */
int
awmh_set_short_payload (int bits)
{
  if (bits == 0)
    {
      Params::payload_short = false;
      Params::payload_size = 128;
      return 0;
    }
  const size_t n = short_code_init (bits);
  if (!n)
    return -1;
  Params::payload_size = bits;
  Params::payload_short = true;
  return int (n);
}

/* --detect-speed / --detect-speed-patient / --try-speed / --test-speed of `audiowmark get` (src/audiowmark.cc:831-854) */
void
awmh_set_speed_params (int detect_speed, int detect_speed_patient, double try_speed, double test_speed)
{
  Params::detect_speed = detect_speed != 0;
  Params::detect_speed_patient = detect_speed_patient != 0;
  Params::try_speed = try_speed;
  Params::test_speed = test_speed;
}

/* detect_speed (src/wmspeed.cc:622-781) for one key on one chunk: best speed / quality as the reference would print
 * them, *accepted = 1 if the speed would be used for a second decode */
int
awmh_detect_speed (const unsigned char *key16, const float *pcm, size_t n_frames, int n_channels, int sample_rate,
                   double *speed, double *quality, int *accepted)
{
  DetectSpeedInfo info;
  const std::vector<DetectSpeedResult> r = detect_speed ({ make_key (key16, "") }, pcm, n_frames, n_channels, sample_rate, false, &info);
  if (!info.valid)
    return 1;
  if (speed)
    *speed = info.speed;
  if (quality)
    *quality = info.quality;
  if (accepted)
    *accepted = r.empty() ? 0 : 1;
  return 0;
}

/* resample_ratio (src/resample.cc:127-131) / the streaming frame count of BufferedResamplerImpl */
int
awmh_resample (const float *in, size_t n_in, int n_channels, double ratio, float *out, size_t n_out)
{
  awm_ctx *ctx = Engine::ctx();
  if (!ctx)
    return 1;
  if (awm_resample (ctx, in, n_in, n_channels, ratio, 16, out, n_out))
    {
      error ("audiowmark: %s\n", awm_last_error (ctx));
      return 1;
    }
  return 0;
}

uint64_t awmh_resample_stream_frames (uint64_t n_in, double ratio) { return resample_stream_frames (n_in, ratio); }
uint64_t awmh_resample_stream_available (uint64_t fed, double ratio) { return resample_stream_available (fed, ratio); }

void
awmh_resampled_add_plan (uint64_t n_frames, int sample_rate, uint64_t *n_emit, uint64_t *gen_runs)
{
  size_t e = 0, r = 0;
  resampled_add_plan (n_frames, sample_rate, !Params::test_no_limiter, sample_rate * int (Params::limiter_block_size_ms) / 1000, e, r);
  *n_emit = e;
  *gen_runs = r;
}

int awmh_frames_per_block() { return int (frames_per_block()); }
int awmh_n_coded_bits()     { return int (code_size (ConvBlockType::a, Params::payload_size)); }

int
awmh_random_u64 (const unsigned char *key16, uint64_t seed, int stream, uint64_t *out, int n)
{
  Random r (make_key (key16, ""), seed, Random::Stream (stream));
  for (int i = 0; i < n; i++)
    out[i] = r();
  return 0;
}

int
awmh_gen_noise (const unsigned char *key16, float *out, size_t n_values)
{
  Random r (make_key (key16, ""), 0, Random::Stream::data_up_down);
  for (size_t i = 0; i < n_values; i++)
    out[i] = r.random_double() * 2 - 1;
  return 0;
}

int
awmh_sync_table (const unsigned char *key16, int mode, awm_sync_entry *out, int max_entries, int *bit_offsets /* [sync_bits + 1] */)
{
  const SyncTable t = gen_sync_table (make_key (key16, ""), mode);
  if (int (t.entries.size()) > max_entries)
    return -1;
  memcpy (out, t.entries.data(), t.entries.size() * sizeof (awm_sync_entry));
  memcpy (bit_offsets, t.bit_offsets.data(), t.bit_offsets.size() * sizeof (int));
  return int (t.entries.size());
}

int
awmh_mix_table (const unsigned char *key16, awm_mix_entry *out, int max_entries, uint16_t *order, int max_order)
{
  const Key key = make_key (key16, "");
  const std::vector<MixEntry> mix = gen_mix_entries (key);
  const std::vector<unsigned> ord = bit_order (key, code_size (ConvBlockType::a, Params::payload_size));
  if (int (mix.size()) > max_entries || int (ord.size()) > max_order)
    return -1;
  for (size_t i = 0; i < mix.size(); i++)
    {
      out[i].frame = mix[i].frame;
      out[i].up = mix[i].up;
      out[i].down = mix[i].down;
    }
  for (size_t i = 0; i < ord.size(); i++)
    order[i] = ord[i];
  return int (mix.size());
}

int
awmh_frame_mod (const unsigned char *key16, const char *payload_hex, uint8_t *out, size_t out_size)
{
  const std::vector<int> bitvec = parse_payload (payload_hex);
  if (bitvec.empty())
    return -1;
  const std::vector<uint8_t> fm = gen_frame_mod_ab (make_key (key16, ""), bitvec);
  if (fm.size() > out_size)
    return -1;
  memcpy (out, fm.data(), fm.size());
  return int (fm.size());
}

int
awmh_conv_encode (int block_type, const uint8_t *bits, int n, uint8_t *out, int max_out)
{
  std::vector<int> in (bits, bits + n);
  const std::vector<int> enc = conv_encode (ConvBlockType (block_type), in);
  if (int (enc.size()) > max_out)
    return -1;
  for (size_t i = 0; i < enc.size(); i++)
    out[i] = enc[i];
  return int (enc.size());
}

/* short payload block code (src/shortcode.cc:136-213) under the current --short setting: encode k -> n bits, decode n -> k bits
 * (returns 0 when no code word matches) */
int
awmh_short_encode (const uint8_t *bits, int k, uint8_t *out, int max_out)
{
  if (!Params::payload_short || size_t (k) != Params::payload_size)
    return -1;
  const std::vector<int> enc = short_encode_blk (std::vector<int> (bits, bits + k));
  if (int (enc.size()) > max_out)
    return -1;
  for (size_t i = 0; i < enc.size(); i++)
    out[i] = enc[i];
  return int (enc.size());
}

int
awmh_short_decode (const uint8_t *coded, int n, uint8_t *out, int max_out)
{
  if (!Params::payload_short || size_t (n) != code_message_bits())
    return -1;
  const std::vector<int> dec = short_decode_blk (std::vector<int> (coded, coded + n));
  if (int (dec.size()) > max_out)
    return -1;
  for (size_t i = 0; i < dec.size(); i++)
    out[i] = dec[i];
  return int (dec.size());
}

/* add_stream_watermark on buffers (host or device pointers) */
int
awmh_add (const unsigned char *key16, const float *in, float *out, size_t n_frames, int n_channels, int sample_rate,
          const char *payload_hex, int *data_blocks, double *snr_db, uint64_t first_frame_number)
{
  AddStats stats;
  const int rc = add_watermark_buffer (make_key (key16, ""), in, out, n_frames, n_channels, sample_rate, payload_hex,
                                       (data_blocks || snr_db) ? &stats : nullptr, first_frame_number);
  if (data_blocks)
    *data_blocks = stats.data_blocks;
  if (snr_db)
    *snr_db = stats.snr_db;
  return rc;
}

/* add / get between 16 bit PCM host buffers (the contents of a 16 bit WAV file): conversions run on the device */
int
awmh_add_s16 (const unsigned char *key16, const int16_t *in, int16_t *out, size_t n_frames, int n_channels, int sample_rate,
              const char *payload_hex, int *data_blocks, double *snr_db, uint64_t first_frame_number)
{
  AddStats stats;
  const int rc = add_watermark_buffer_s16 (make_key (key16, ""), in, out, n_frames, n_channels, sample_rate, payload_hex, (data_blocks || snr_db) ? &stats : nullptr,
                                           first_frame_number);
  if (data_blocks)
    *data_blocks = stats.data_blocks;
  if (snr_db)
    *snr_db = stats.snr_db;
  return rc;
}

/* add_stream_watermark's bounded-memory loop (add_watermark_windowed) between two host buffers: `in` is read in small blocks like a
 * pipe, the result is appended to `out` (n_frames frames); window_frames = 0 uses the default window.  zero_frames: the input continues
 * a stream that began that many frames earlier with silence (src/wmadd.cc:504-519). */
int
awmh_add_windowed (const unsigned char *key16, const float *in, float *out, size_t n_frames, int n_channels, int sample_rate, const char *payload_hex,
                   size_t zero_frames, size_t window_frames, int *data_blocks, double *snr_db)
{
  size_t rpos = 0, wpos = 0;
  auto read = [&] (std::vector<float>& samples, size_t count)
    {
      const size_t n = std::min (count, n_frames - rpos);
      samples.assign (in + rpos * n_channels, in + (rpos + n) * n_channels);
      rpos += n;
      return Error (Error::Code::NONE);
    };
  auto write = [&] (const std::vector<float>& samples)
    {
      if (wpos * n_channels + samples.size() > n_frames * n_channels)
        return Error ("output buffer too small");
      memcpy (out + wpos * n_channels, samples.data(), samples.size() * sizeof (float));
      wpos += samples.size() / n_channels;
      return Error (Error::Code::NONE);
    };
  AddStats stats;
  size_t written = 0;
  const int rc = add_watermark_windowed (make_key (key16, ""), read, write, n_channels, sample_rate, payload_hex, zero_frames, window_frames, &stats, &written);
  if (rc)
    return rc;
  if (data_blocks) *data_blocks = stats.data_blocks;
  if (snr_db) *snr_db = stats.snr_db;
  return written == n_frames ? 0 : -3;
}

static int result_json (ResultSet& result_set, size_t mark_rate_frames, char *json_out, size_t json_cap, int *n_patterns);

int
awmh_get_s16 (const unsigned char *keys16, const char *const *names, int n_keys, const int16_t *pcm, size_t n_frames, int n_channels,
              int sample_rate, char *json_out, size_t json_cap, int *n_patterns)
{
  std::vector<Key> key_list;
  for (int k = 0; k < n_keys; k++)
    key_list.push_back (make_key (keys16 + 16 * k, names ? names[k] : ""));
  ResultSet result_set;
  size_t mark_rate_frames = n_frames;
  const int rc = get_watermark_buffer_s16 (key_list, pcm, n_frames, n_channels, sample_rate, result_set, false, &mark_rate_frames);
  if (rc)
    return rc;
  return result_json (result_set, mark_rate_frames, json_out, json_cap, n_patterns);
}

/* `get` on the stored sample bytes of a WAV file held in memory (n_bytes / (bits / 8 * n_channels) frames; 8 bit is unsigned as in
 * WAV): at 44.1 kHz the streamed loader of the CLI runs over the buffer (get_watermark_stream; two page-locked chunk buffers, decoded
 * on the device), piece_frames frames per read of the buffer (0: a chunk per read); other rates are converted on the host and
 * resampled as a whole, as the CLI does.  Writes the --json document into json_out. */
int
awmh_get_wav (const unsigned char *keys16, const char *const *names, int n_keys, const unsigned char *data, size_t n_bytes, int n_channels,
              int bits, int is_float, int sample_rate, size_t piece_frames, char *json_out, size_t json_cap, int *n_patterns)
{
  if (n_channels <= 0 || (bits != 8 && bits != 16 && bits != 24 && bits != 32 && bits != 64))
    return 1;
  std::vector<Key> key_list;
  for (int k = 0; k < n_keys; k++)
    key_list.push_back (make_key (keys16 + 16 * k, names ? names[k] : ""));
  const size_t frame_bytes = size_t (bits / 8) * n_channels, n_frames = n_bytes / frame_bytes;
  ResultSet result_set;
  size_t mark_rate_frames = n_frames;
  if (sample_rate == Params::mark_sample_rate)
    {
      size_t pos = 0;
      auto source = [&] (unsigned char *dst, size_t count, size_t *n_read)
        {
          *n_read = std::min (count, n_frames - pos);
          memcpy (dst, data + pos * frame_bytes, *n_read * frame_bytes);
          pos += *n_read;
          return Error (Error::Code::NONE);
        };
      Error read_err;
      const int rc = get_watermark_stream (key_list, source, awm_wav_format { bits, is_float ? 1 : 0 }, n_channels, n_frames, piece_frames, result_set,
                                           false, &mark_rate_frames, read_err);
      if (rc)
        return rc;
    }
  else
    {
      RawFormat format (n_channels, sample_rate, bits);
      format.set_encoding (is_float ? Encoding::FLOAT : bits == 8 ? Encoding::UNSIGNED : Encoding::SIGNED);
      Error err;
      std::unique_ptr<RawConverter> conv (RawConverter::create (format, err));
      if (err)
        return 1;
      std::vector<float> samples (n_frames * n_channels);
      conv->from_raw (data, samples.data(), samples.size());
      const int rc = get_watermark_buffer (key_list, samples.data(), n_frames, n_channels, sample_rate, result_set, false, &mark_rate_frames);
      if (rc)
        return rc;
    }
  return result_json (result_set, mark_rate_frames, json_out, json_cap, n_patterns);
}

/* test aid (CPU): RawConverter::from_raw of n_samples stored WAV samples (8 bit unsigned, 16/24/32 bit signed, 32/64 bit float,
 * little endian), the host conversion the device decode (awm_pcm_bind_wav) must equal bit for bit */
int
awmh_wav_decode_host (const unsigned char *bytes, size_t n_samples, int bits, int is_float, float *out)
{
  RawFormat format (1, Params::mark_sample_rate, bits);
  format.set_encoding (is_float ? Encoding::FLOAT : bits == 8 ? Encoding::UNSIGNED : Encoding::SIGNED);
  Error err;
  std::unique_ptr<RawConverter> conv (RawConverter::create (format, err));
  if (err)
    return 1;
  conv->from_raw (bytes, out, n_samples);
  return 0;
}

/* get_watermark on a buffer (host pointer; a device pointer is accepted for inputs longer than 3.1 blocks,
 * where the clip decoder is not used).  Writes the --json document into json_out. */
int
awmh_get (const unsigned char *keys16, const char *const *names, int n_keys, const float *pcm, size_t n_frames, int n_channels,
          int sample_rate, char *json_out, size_t json_cap, int *n_patterns)
{
  std::vector<Key> key_list;
  for (int k = 0; k < n_keys; k++)
    key_list.push_back (make_key (keys16 + 16 * k, names ? names[k] : ""));
  ResultSet result_set;
  size_t mark_rate_frames = n_frames;
  const int rc = get_watermark_buffer (key_list, pcm, n_frames, n_channels, sample_rate, result_set, false, &mark_rate_frames);
  if (rc)
    return rc;
  return result_json (result_set, mark_rate_frames, json_out, json_cap, n_patterns);
}

static int
result_json (ResultSet& result_set, size_t mark_rate_frames, char *json_out, size_t json_cap, int *n_patterns)
{
  if (n_patterns)
    *n_patterns = int (result_set.all().size());
  if (json_out && json_cap)
    {
      char *buf = nullptr;
      size_t len = 0;
      FILE *f = open_memstream (&buf, &len);
      result_set.print_json (f, size_t (lrint (double (mark_rate_frames) / Params::mark_sample_rate)));
      fclose (f);
      if (len + 1 > json_cap)
        {
          free (buf);
          return -2;
        }
      memcpy (json_out, buf, len + 1);
      free (buf);
    }
  return 0;
}

/* ---- sharded `get`: chunk results as flat records ------------------------------------------------
 * record (little endian, packed): i32 key_index, f64 time, f64 quality, u64 sync_index, f32 decode_error,
 * u8 block_type, u8 type, f64 speed, u16 n_bits, n_bits bytes (0/1)
 */
static void
put (std::vector<unsigned char>& b, const void *p, size_t n)
{
  const unsigned char *c = static_cast<const unsigned char *> (p);
  b.insert (b.end(), c, c + n);
}

static std::vector<unsigned char>
serialize (const ResultSet& rs, const std::vector<Key>& key_list)
{
  std::vector<unsigned char> b;
  for (const auto& p : rs.all())
    {
      int32_t ki = 0;
      for (size_t k = 0; k < key_list.size(); k++)
        if (key_list[k] == p.key)
          ki = k;
      const double time = p.time, quality = p.sync_score.quality, speed = p.speed;
      const uint64_t idx = p.sync_score.index;
      const float err = p.decode_error;
      const uint8_t bt = uint8_t (p.sync_score.block_type), ty = uint8_t (p.type);
      const uint16_t nb = p.bit_vec.size();
      put (b, &ki, 4); put (b, &time, 8); put (b, &quality, 8); put (b, &idx, 8); put (b, &err, 4);
      put (b, &bt, 1); put (b, &ty, 1); put (b, &speed, 8); put (b, &nb, 2);
      for (int bit : p.bit_vec)
        b.push_back (bit ? 1 : 0);
    }
  return b;
}

static bool
deserialize (const unsigned char *b, size_t len, const std::vector<Key>& key_list, ResultSet& rs)
{
  size_t pos = 0;
  auto get = [&] (void *p, size_t n) { if (pos + n > len) return false; memcpy (p, b + pos, n); pos += n; return true; };
  while (pos < len)
    {
      int32_t ki; double time, quality, speed; uint64_t idx; float err; uint8_t bt, ty; uint16_t nb;
      if (!get (&ki, 4) || !get (&time, 8) || !get (&quality, 8) || !get (&idx, 8) || !get (&err, 4) || !get (&bt, 1) || !get (&ty, 1)
          || !get (&speed, 8) || !get (&nb, 2) || pos + nb > len || ki < 0 || size_t (ki) >= key_list.size() || bt > 2 || ty > 2)
        return false;
      std::vector<int> bits (b + pos, b + pos + nb);
      pos += nb;
      rs.add_pattern (key_list[ki], time, SyncFinder::Score { size_t (idx), quality, ConvBlockType (bt) }, bits, err, ResultSet::Type (ty), speed);
    }
  return true;
}

static std::vector<Key>
make_key_list (const unsigned char *keys16, const char *const *names, int n_keys)
{
  std::vector<Key> key_list;
  for (int k = 0; k < n_keys; k++)
    key_list.push_back (make_key (keys16 + 16 * k, names ? names[k] : ""));
  return key_list;
}

/* decode ONE chunk of the reference's chunk geometry (pcm = the chunk's samples); records -> blob_out */
int
awmh_get_chunk (const unsigned char *keys16, const char *const *names, int n_keys, const float *pcm, size_t n_frames, int n_channels,
                int sample_rate, int first_chunk, unsigned char *blob_out, size_t blob_cap, size_t *blob_len)
{
  const std::vector<Key> key_list = make_key_list (keys16, names, n_keys);
  ResultSet rs;
  const int rc = get_watermark_chunk (key_list, pcm, n_frames, n_channels, sample_rate, first_chunk != 0, rs);
  if (rc)
    return rc;
  const std::vector<unsigned char> b = serialize (rs, key_list);
  *blob_len = b.size();
  if (b.size() > blob_cap)
    return -2;
  if (!b.empty())
    memcpy (blob_out, b.data(), b.size());
  return 0;
}

/* ResultSet::merge in chunk order + sort + --json document (src/wmget.cc:289-316,252-287,340-382) from chunk blobs */
int
awmh_merge_chunks (const unsigned char *keys16, const char *const *names, int n_keys, const unsigned char *const *blobs, const size_t *blob_lens,
                   const double *time_offsets, int n_chunks, double total_seconds, char *json_out, size_t json_cap)
{
  const std::vector<Key> key_list = make_key_list (keys16, names, n_keys);
  ResultSet result_set;
  for (int c = 0; c < n_chunks; c++)
    {
      ResultSet chunk;
      if (!deserialize (blobs[c], blob_lens[c], key_list, chunk))
        return -3;
      chunk.apply_time_offset (time_offsets[c]);
      result_set.merge (chunk);
    }
  result_set.sort (key_list);
  char *buf = nullptr;
  size_t len = 0;
  FILE *f = open_memstream (&buf, &len);
  result_set.print_json (f, size_t (lrint (total_seconds)));
  fclose (f);
  const bool fits = len + 1 <= json_cap;
  if (fits)
    memcpy (json_out, buf, len + 1);
  free (buf);
  return fits ? 0 : -2;
}

void
awmh_chunk_geometry (int sample_rate, uint64_t *max_frames, uint64_t *overlap_frames)
{
  size_t m, o;
  chunk_geometry (sample_rate, m, o);
  *max_frames = m;
  *overlap_frames = o;
}

/* ---- sharded `get`: one long stream over several GPUs (awm_balanced.hh) --------------------------------------------------- */

int
awmh_dist_unique_id (unsigned char id_out[128])
{
  return awm_dist_unique_id (id_out);
}

/* join the NCCL communicator of the job (the id comes from rank 0's awmh_dist_unique_id, handed round by the launcher) */
int
awmh_dist_init (int rank, int world, const unsigned char id[128])
{
  awm_ctx *ctx = Engine::ctx();
  if (!ctx)
    return 1;
  if (awm_dist_init (ctx, rank, world, id))
    {
      error ("audiowmark: %s\n", awm_last_error (ctx));
      return 1;
    }
  return 0;
}

/* every rank calls this with its part of the stream ([pcm_start, pcm_start + pcm_frames) of n_total frames; float or 16 bit PCM,
 * host or device memory); rank 0 receives the --json document (n_patterns >= 0), the other ranks n_patterns = -1 */
int
awmh_balanced_get (const unsigned char *key16, const void *pcm, int is_s16, uint64_t pcm_start, uint64_t pcm_frames, uint64_t n_total, int n_channels,
                   int sample_rate, char *json_out, size_t json_cap, int *n_patterns)
{
  awm_ctx *ctx = Engine::ctx();
  if (!ctx)
    return 1;
  int rank = 0, world = 1;
  awm_dist_world (ctx, &rank, &world);
  balanced::Get job (rank, world, n_total, is_s16 ? nullptr : static_cast<const float *> (pcm), is_s16 ? static_cast<const int16_t *> (pcm) : nullptr,
                     pcm_start, pcm_frames, n_channels, sample_rate, make_key (key16, ""));
  if (!job.ok())
    return 1;
  std::vector<unsigned char> recv;
  std::vector<size_t> lens (world);
  /* bytes per rank in an exchange: the refined scores + soft bits of a rank's candidates are ~0.4 MB per hour of audio; a payload that
   * does not fit costs a second round, so the size that was needed once is kept for the following calls */
  static size_t slot = 1024 * 1024;
  auto exchange = [&] (const std::string& mine, std::vector<std::string>& all)
    {
      for (;;)
        {
          recv.resize (slot * world);
          const int rc = awm_dist_allgather (ctx, mine.data(), mine.size(), slot, recv.data(), lens.data());
          if (rc == 2)                               // somebody's payload did not fit: every rank saw the same lengths
            {
              slot = (*std::max_element (lens.begin(), lens.end()) + 8 + 4095) / 4096 * 4096;
              continue;
            }
          if (rc)
            {
              error ("audiowmark: %s\n", awm_last_error (ctx));
              return false;
            }
          break;
        }
      all.resize (world);
      for (int r = 0; r < world; r++)
        all[r].assign (reinterpret_cast<const char *> (recv.data()) + size_t (r) * slot, lens[r]);
      return true;
    };
  ResultSet result_set;
  if (!job.run (exchange, result_set))
    return 1;
  if (rank != 0)
    {
      if (n_patterns)
        *n_patterns = -1;
      return 0;
    }
  return result_json (result_set, n_total, json_out, json_cap, n_patterns);
}

/* the stages one by one, for tests that run several ranks in one process on one GPU (tests/test_gpu_sharding.py):
 * stage 0 peaks, 1 select (-> retry list), 2 peaks again for the retry list in in[0], 3 refine + soft bits, 4 viterbi, 5 merge (-> JSON) */
void *
awmh_bg_create (const unsigned char *key16, int rank, int world, const float *pcm, uint64_t pcm_start, uint64_t pcm_frames, uint64_t n_total, int n_channels, int sample_rate)
{
  balanced::Get *g = new balanced::Get (rank, world, n_total, pcm, nullptr, pcm_start, pcm_frames, n_channels, sample_rate, make_key (key16, ""));
  if (!g->ok())
    {
      delete g;
      return nullptr;
    }
  return g;
}

void
awmh_bg_destroy (void *h)
{
  delete static_cast<balanced::Get *> (h);
}

int
awmh_bg_stage (void *h, int stage, const unsigned char *const *in, const size_t *in_len, int n_in, uint64_t n_total, unsigned char *out, size_t cap, size_t *out_len)
{
  balanced::Get *g = static_cast<balanced::Get *> (h);
  std::vector<std::string> all;
  for (int i = 0; i < n_in; i++)
    all.emplace_back (reinterpret_cast<const char *> (in[i]), in_len[i]);
  std::string res;
  bool ok = false;
  auto parse_floors = [] (const std::string& s)
    {
      std::map<int, double> m;
      for (size_t pos = 0; pos + 12 <= s.size(); pos += 12)
        {
          int32_t c; double f;
          memcpy (&c, s.data() + pos, 4); memcpy (&f, s.data() + pos + 4, 8);
          m[c] = f;
        }
      return m;
    };
  switch (stage)
    {
    case 0: ok = g->stage_peaks ({}, res); break;
    case 1:
      {
        std::map<int, double> retry;
        ok = g->stage_select (all, retry);
        for (const auto& kv : retry)
          {
            const int32_t c = kv.first; const double f = kv.second;
            res.append (reinterpret_cast<const char *> (&c), 4);
            res.append (reinterpret_cast<const char *> (&f), 8);
          }
        break;
      }
    case 2: ok = g->stage_peaks (parse_floors (all.empty() ? std::string() : all[0]), res); break;
    case 3: ok = g->stage_refine_decode (res); break;
    case 4: ok = g->stage_viterbi (all, res); break;
    case 5:
      {
        ResultSet rs;
        ok = g->stage_merge (all, rs);
        if (ok)
          {
            char *buf = nullptr;
            size_t len = 0;
            FILE *f = open_memstream (&buf, &len);
            rs.print_json (f, size_t (lrint (double (n_total) / Params::mark_sample_rate)));
            fclose (f);
            res.assign (buf, len);
            free (buf);
          }
        break;
      }
    }
  if (!ok)
    return 1;
  *out_len = res.size();
  if (res.size() > cap)
    return -2;
  if (!res.empty())
    memcpy (out, res.data(), res.size());
  return 0;
}

/* the plan functions for CPU tests: chunk walk, slices of a rank, owner of an index */
int
awmh_bg_plan (uint64_t n_total, int sample_rate, int rank, int world, double *chunks /* [max][3] first, count, time offset */, int max_chunks, int *n_chunks,
              int64_t *slices /* [max][7] chunk, sa, sb, a, b, lo, hi */, int max_slices, int *n_slices)
{
  const auto plan = balanced::chunk_plan (n_total, sample_rate);
  *n_chunks = int (plan.size());
  for (int c = 0; c < int (plan.size()) && c < max_chunks; c++)
    {
      chunks[3 * c] = double (plan[c].first);
      chunks[3 * c + 1] = double (plan[c].count);
      chunks[3 * c + 2] = plan[c].time_offset;
    }
  const auto sl = balanced::rank_slices (plan, rank, world, n_total);
  *n_slices = int (sl.size());
  for (int i = 0; i < int (sl.size()) && i < max_slices; i++)
    {
      const int64_t v[7] = { sl[i].chunk, sl[i].sa, sl[i].sb, sl[i].a, sl[i].b, int64_t (sl[i].lo), int64_t (sl[i].hi) };
      memcpy (slices + 7 * i, v, sizeof (v));
    }
  return 0;
}

int
awmh_bg_owner (uint64_t n_total, int sample_rate, int world, int chunk, uint64_t index)
{
  return balanced::owner_of (balanced::chunk_plan (n_total, sample_rate), n_total, world, chunk, index);
}

/* ---- stage-level access for the frame-balanced multi-GPU driver (audiowmark_b200/sharding.py) ---------------- */

void *
awmh_ctx()
{
  return Engine::ctx();
}

int
awmh_key_slot (const unsigned char *key16)
{
  return Engine::key_slot (make_key (key16, ""));
}

/* test aid (CPU): ResultSet::merge and ResultSet::sort against their literal definitions (src/wmget.cc:268-312: scan everything found so
 * far with approx_match; compare name / rating / all-last / time / A-B-AB / bits one after the other) on random chunk results: a few
 * payloads, positions that collide within a frame across chunks, combined patterns, stretched speeds, two keys.  Returns 0 when the
 * merged and sorted documents are identical, else the number of the first failing round + 1. */
int
awmh_selftest_results (uint64_t seed, int rounds)
{
  uint64_t state = seed * 6364136223846793005ull + 1442695040888963407ull;
  auto rnd = [&] (uint32_t n) { state = state * 6364136223846793005ull + 1442695040888963407ull; return uint32_t ((state >> 33) % n); };
  const double frame = Params::frame_size / double (Params::mark_sample_rate);
  Key keys[2];
  keys[0] = make_key (reinterpret_cast<const unsigned char *> ("0123456789abcdef"), "alpha");
  keys[1] = make_key (reinterpret_cast<const unsigned char *> ("fedcba9876543210"), "beta");
  size_t n_in = 0, n_kept = 0;
  for (int round = 0; round < rounds; round++)
    {
      std::vector<std::vector<int>> payloads (3 + rnd (3), std::vector<int> (16));
      for (auto& pl : payloads)
        for (int& b : pl)
          b = int (rnd (2));
      const int n_chunks = 2 + int (rnd (4));
      std::vector<ResultSet> chunks (n_chunks), chunks_copy;
      for (int c = 0; c < n_chunks; c++)
        for (int i = 0, n = int (rnd (40)); i < n; i++)
          {
            const ResultSet::Type type = rnd (10) == 0 ? ResultSet::Type::ALL : rnd (8) == 0 ? ResultSet::Type::CLIP : ResultSet::Type::BLOCK;
            const ConvBlockType bt = ConvBlockType (rnd (3));
            /* positions on a coarse grid + a jitter around one frame, so that patterns of neighbouring chunks fall inside and just outside the match window */
            /* + a unique 1e-7 s: no two patterns tie in every sort key (std::sort leaves the order of ties open, in the reference too) */
            const double time = double (rnd (12)) * 7.0 + (double (rnd (5)) - 2.0) * frame * 0.6 + 1e-7 * double (c * 64 + i);
            const double speed = rnd (6) == 0 ? 1.0 + (double (rnd (5)) - 2.0) * 0.006 : 1.0;
            chunks[c].add_pattern (keys[rnd (2)], time, SyncFinder::Score { size_t (rnd (100000)), double (rnd (1000)) / 1000.0, bt }, payloads[rnd (uint32_t (payloads.size()))],
                                   float (rnd (100)) / 100.f, type, speed);
          }
      chunks_copy = chunks;
      /* the library */
      ResultSet merged;
      for (int c = 0; c < n_chunks; c++)
        {
          chunks[c].apply_time_offset (0.4 * frame * c);
          merged.merge (chunks[c]);
        }
      merged.sort ({ keys[0], keys[1] });
      /* the definition */
      std::vector<ResultSet::Pattern> ref;
      for (int c = 0; c < n_chunks; c++)
        {
          chunks_copy[c].apply_time_offset (0.4 * frame * c);
          std::vector<ResultSet::Pattern> in = chunks_copy[c].all();
          std::stable_sort (in.begin(), in.end(), [] (const ResultSet::Pattern& a, const ResultSet::Pattern& b) { return a.time < b.time; });
          for (const auto& p : in)
            {
              bool is_new = true;
              for (const auto& have : ref)
                if (have.approx_match (p))
                  is_new = false;
              if (is_new)
                ref.push_back (p);
            }
        }
      for (const Key& key : keys)
        {
          std::map<std::string, float> rating;
          for (const auto& p : ref)
            if (p.key == key)
              rating[bit_vec_to_str (p.bit_vec)] += p.sync_score.quality * (p.type == ResultSet::Type::ALL ? 2.f : 1.f);
          for (auto& p : ref)
            if (p.key == key)
              p.rating = rating[bit_vec_to_str (p.bit_vec)];
        }
      auto rank_of = [] (const ResultSet::Pattern& p) { return p.sync_score.block_type == ConvBlockType::a ? 0 : p.sync_score.block_type == ConvBlockType::b ? 1 : 2; };
      std::sort (ref.begin(), ref.end(), [&] (const ResultSet::Pattern& a, const ResultSet::Pattern& b)
        {
          const int all_a = a.type == ResultSet::Type::ALL, all_b = b.type == ResultSet::Type::ALL;
          if (a.key.name() != b.key.name()) return a.key.name() < b.key.name();
          if (a.rating != b.rating) return a.rating > b.rating;
          if (all_a != all_b) return all_a < all_b;
          if (a.time != b.time) return a.time < b.time;
          if (rank_of (a) != rank_of (b)) return rank_of (a) < rank_of (b);
          return bit_vec_to_str (a.bit_vec) < bit_vec_to_str (b.bit_vec);
        });
      const auto& got = merged.all();
      bool same = got.size() == ref.size();
      for (size_t i = 0; same && i < ref.size(); i++)
        same = got[i].key == ref[i].key && got[i].time == ref[i].time && got[i].bit_vec == ref[i].bit_vec && got[i].type == ref[i].type
            && got[i].sync_score.block_type == ref[i].sync_score.block_type && got[i].sync_score.quality == ref[i].sync_score.quality
            && got[i].speed == ref[i].speed && got[i].rating == ref[i].rating && got[i].decode_error == ref[i].decode_error;
      if (!same)
        return round + 1;
      for (const ResultSet& cr : chunks_copy)
        n_in += cr.all().size();
      n_kept += ref.size();
    }
  /* the test has teeth only if the merge did drop detections and keep others */
  return (n_kept < n_in && n_kept * 10 > n_in) ? 0 : -1;
}

/* test aid: sync positions.  awmh_sync_trace (1) starts recording what every SyncFinder::search call returns, awmh_sync_trace_fetch
 * copies the records out as rows of 5 doubles {search number, mode (0 BLOCK / 1 CLIP), searched frames, -1, -1} (one header row per
 * search) and {search number, index, quality, block type (0 A / 1 B), 0} (one row per score) and clears the trace */
int
awmh_sync_trace (int on)
{
  SyncFinder::trace_enable (on != 0);
  return 0;
}

int
awmh_sync_trace_fetch (double *rows, size_t max_rows, size_t *n_rows)
{
  const auto trace = SyncFinder::trace_take();
  size_t n = 0;
  auto put = [&] (double a, double b, double c, double d, double e)
    {
      if (n < max_rows)
        {
          double *r = rows + 5 * n;
          r[0] = a; r[1] = b; r[2] = c; r[3] = d; r[4] = e;
        }
      n++;
    };
  for (size_t i = 0; i < trace.size(); i++)
    {
      put (double (i), trace[i].mode == SyncFinder::Mode::CLIP ? 1 : 0, double (trace[i].n_frames), -1, -1);
      for (const auto& sc : trace[i].scores)
        put (double (i), double (sc.index), sc.quality, sc.block_type == ConvBlockType::a ? 0 : 1, 0);
    }
  *n_rows = n;
  return n <= max_rows ? 0 : -2;
}

/* candidates of one chunk from its (gathered) peak list, complete above floor_q; *complete = 0 -> ask again with a lower floor */
int
awmh_stage_select (const awm_search_score *peaks, size_t n, double floor_q, int clip_mode, awm_search_score *out, size_t max_out, size_t *n_out, int *complete)
{
  std::vector<awm_search_score> sel;
  *complete = select_candidates_from_peaks (peaks, n, floor_q, Params::sync_threshold2 * 0.75, sel) > 0 ? 1 : 0;
  if (clip_mode)
    {
      std::sort (sel.begin(), sel.end(), [] (const awm_search_score& a, const awm_search_score& b) { return fabs (a.raw_quality - a.local_mean) > fabs (b.raw_quality - b.local_mean); });
      const size_t n_max = std::max (Params::get_n_best, 5);
      if (sel.size() > n_max)
        sel.resize (n_max);
    }
  *n_out = sel.size();
  if (sel.size() > max_out)
    return -2;
  if (!sel.empty())
    memcpy (out, sel.data(), sel.size() * sizeof (awm_search_score));
  return 0;
}

/* threshold2 / n-best selection of a chunk's refined scores -> (index, quality, block type) sorted by index */
int
awmh_stage_final (const awm_search_score *refined, size_t n, uint64_t *index_out, double *quality_out, int *btype_out, size_t *n_out)
{
  std::vector<awm_search_score> v (refined, refined + n);
  std::vector<SyncFinder::Score> out;
  select_final_scores (v, out);
  *n_out = out.size();
  for (size_t i = 0; i < out.size(); i++)
    {
      index_out[i] = out[i].index;
      quality_out[i] = out[i].quality;
      btype_out[i] = int (out[i].block_type);
    }
  return 0;
}

/* Viterbi job list (single blocks, AB pairs, "all") of one chunk from its final scores and their soft bits */
int
awmh_stage_jobs (const unsigned char *key16, const uint64_t *index, const double *quality, const int *btype, size_t n, const float *raw, const int *valid,
                 int sample_rate, unsigned char *blob, size_t cap, size_t *len, int *n_jobs)
{
  const size_t n_coded = code_size (ConvBlockType::a, Params::payload_size);
  std::vector<SyncFinder::Score> scores (n);
  std::vector<std::vector<float>> rawv (n);
  std::vector<int> validv (valid, valid + n);
  for (size_t i = 0; i < n; i++)
    {
      scores[i] = SyncFinder::Score { size_t (index[i]), quality[i], ConvBlockType (btype[i]) };
      rawv[i].assign (raw + i * n_coded, raw + (i + 1) * n_coded);
    }
  const std::vector<unsigned char> b = block_jobs_blob (make_key (key16, ""), scores, rawv, validv, sample_rate, n_jobs);
  *len = b.size();
  if (b.size() > cap)
    return -2;
  if (!b.empty())
    memcpy (blob, b.data(), b.size());
  return 0;
}

uint64_t
awmh_gpu_launches()
{
  awm_ctx *c = Engine::ctx();
  return c ? awm_launch_count (c) : 0;
}

void *
awmh_gpu_stream()
{
  awm_ctx *c = Engine::ctx();
  return c ? awm_stream (c) : nullptr;
}

/* device-pointer calls are stream ordered and return without waiting: synchronise before touching the results from
 * another stream / the host */
int
awmh_synchronize()
{
  awm_ctx *c = Engine::ctx();
  return c ? awm_synchronize (c) : 1;
}

int
awmh_profile_enable (int on)
{
  awm_ctx *c = Engine::ctx();
  return c ? awm_profile_enable (c, on) : 1;
}

int
awmh_profile_report (char *json_out, size_t cap)
{
  awm_ctx *c = Engine::ctx();
  return c ? awm_profile_report (c, json_out, cap) : 1;
}

void
awmh_shutdown()
{
  Engine::shutdown();
}

} // extern "C"
