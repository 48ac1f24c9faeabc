// awm_get.cc -- `audiowmark get / cmp`: chunk loop, BlockDecoder, ClipDecoder, ResultSet
// (reference src/wmget.cc:163-1013, src/wavchunkloader.cc:54-239).  FFTs, soft-bit extraction and the
// Viterbi decoder run on the GPU through the C ABI; pairing / combining logic stays on the host.
#include "awm_results.hh"
#include "awm_get_internal.hh"
#include "awm_speed.hh"
#include "awm_engine.hh"
#include "awm_tables.hh"
#include "awm_util.hh"

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <map>
#include <math.h>
#include <memory>
#include <mutex>
#include <thread>
#include <string.h>
#include <stdlib.h>

using std::string;
using std::vector;
using std::max;
using std::min;

int
frame_count (const WavData& wav_data)
{
  return wav_data.n_values() / wav_data.n_channels() / Params::frame_size;
}

/* ---------------------------------------------------------------- GPU helpers */

namespace get_detail {

/* code_decode_soft for a set of code words (A, B and AB mixed) in ONE awm_viterbi launch */
bool
viterbi_decode (const vector<const VitJob *>& jobs, vector<uint8_t>& bits, vector<float>& err)
{
  awm_ctx *ctx = Engine::ctx();
  if (!ctx)
    return false;
  const int n_msg = int (code_message_bits());        /* the block code word in short payload mode */
  bits.assign (jobs.size() * n_msg, 0);
  err.assign (jobs.size(), 0.f);
  if (jobs.empty())
    return true;
  vector<float> raw;
  vector<int> types (jobs.size());
  for (size_t j = 0; j < jobs.size(); j++)
    {
      raw.insert (raw.end(), jobs[j]->soft.begin(), jobs[j]->soft.end());
      types[j] = jobs[j]->block_type == ConvBlockType::a ? AWM_BLOCK_A : jobs[j]->block_type == ConvBlockType::b ? AWM_BLOCK_B : AWM_BLOCK_AB;
    }
  if (awm_viterbi (ctx, raw.data(), jobs.size(), n_msg, types.data(), Params::hard ? 1 : 0, bits.data(), err.data()))
    {
      error ("audiowmark: viterbi decoder failed: %s\n", awm_last_error (ctx));
      return false;
    }
  return true;
}

void
add_decoded_pattern (const VitJob& job, const uint8_t *bits, float err, ResultSet& chunk_result)
{
  const int n_msg = int (code_message_bits());
  vector<int> bit_vec (bits, bits + n_msg);
  if (Params::payload_short)
    {
      bit_vec = short_decode_blk (bit_vec);        /* code_decode_soft, src/shortcode.cc:129-133 */
      if (bit_vec.empty())
        return;
    }
  chunk_result.add_pattern (job.key, job.time, job.score, bit_vec, err, job.type, job.speed);
}

/* every pending code word of a `get` run (all chunks and keys) in one launch; the decoded patterns go to the result set of the
 * chunk they came from */
bool
run_viterbi_jobs (vector<VitJob>& jobs, vector<ResultSet>& chunk_results)
{
  vector<const VitJob *> list;
  for (const auto& j : jobs)
    list.push_back (&j);
  vector<uint8_t> bits;
  vector<float> err;
  if (!viterbi_decode (list, bits, err))
    return false;
  const int n_msg = int (code_message_bits());
  for (size_t j = 0; j < jobs.size(); j++)
    add_decoded_pattern (jobs[j], bits.data() + j * n_msg, err[j], chunk_results[jobs[j].chunk]);
  jobs.clear();
  return true;
}

/* fft_range + mix_decode + randomize_bit_order (decode) for several block start positions */
bool
decode_raw_bits (const Key& key, const vector<uint64_t>& indices, vector<vector<float>>& raw, vector<int>& valid)
{
  awm_ctx *ctx = Engine::ctx();
  const int slot = ctx ? Engine::key_slot (key) : -1;
  if (slot < 0)
    return false;
  const size_t n_coded = code_size (ConvBlockType::a, Params::payload_size);
  vector<float> flat (indices.size() * n_coded);
  valid.assign (indices.size(), 0);
  if (awm_decode_blocks (ctx, slot, indices.data(), indices.size(), flat.data(), valid.data()))
    {
      error ("audiowmark: block decode failed: %s\n", awm_last_error (ctx));
      return false;
    }
  raw.resize (indices.size());
  for (size_t i = 0; i < indices.size(); i++)
    raw[i].assign (flat.begin() + i * n_coded, flat.begin() + (i + 1) * n_coded);
  return true;
}

/* What BlockDecoder::run does once the soft bits of the synchronised blocks are known (src/wmget.cc:539-701), as three separate
 * steps over one list of decoded blocks (in sync-score order = ascending position):
 *   single blocks   every valid block is a code word of its own type
 *   AB pairs        a B block together with the A block that starts one block length before it
 *   "all"           the longest-scoring chain of alternating blocks, soft bits averaged per type
 * The selection rules (tolerances, strict comparisons, float accumulation of the chain score) are the reference's: they decide
 * which patterns are printed. */
struct DecodedBlock
{
  size_t               index;
  double               quality;
  ConvBlockType        type;
  const vector<float> *soft;
};

ConvBlockType
other_type (ConvBlockType t)
{
  return t == ConvBlockType::a ? ConvBlockType::b : ConvBlockType::a;
}

/* position in `blocks` of the block of type `want` nearest to sample `target`, among positions >= first and < last, nearer than
 * `tolerance` samples (the earliest of equally near blocks); -1 if there is none */
int
nearest_block (const vector<DecodedBlock>& blocks, size_t first, size_t last, ConvBlockType want, int target, int tolerance)
{
  int found = -1, nearest = tolerance;
  for (size_t j = first; j < last; j++)
    {
      const int dist = std::abs (target - int (blocks[j].index));
      if (blocks[j].type == want && dist < nearest)
        {
          found = int (j);
          nearest = dist;
        }
    }
  return found;
}

/* chain of alternating blocks that starts at block `head`: after the last member, the block expected k block lengths later
 * (type flips with odd k) is looked for with k = 1, 2, ... and a tolerance that grows with k; a hit restarts at k = 1 */
vector<size_t>
alternating_chain (const vector<DecodedBlock>& blocks, size_t head, size_t block_len)
{
  const size_t k_max = lrint (blocks.back().index / double (block_len) + 0.5);
  vector<size_t> chain { head };
  for (size_t k = 1; k <= k_max; )
    {
      const DecodedBlock& tail = blocks[chain.back()];
      const int next = nearest_block (blocks, chain.back(), blocks.size(), (k & 1) ? other_type (tail.type) : tail.type,
                                      int (tail.index + k * block_len), int (k * Params::frame_size / 2));
      if (next >= 0)
        {
          chain.push_back (next);
          k = 1;
        }
      else
        k++;
    }
  return chain;
}

float
chain_score (const vector<DecodedBlock>& blocks, const vector<size_t>& chain)
{
  float sum = 0;                                  /* single precision like the reference: it breaks near ties the same way */
  for (size_t b : chain)
    sum += blocks[b].quality;
  return sum;
}

void
build_block_jobs (const Key& key, const vector<SyncFinder::Score>& sync_scores, const vector<vector<float>>& raw, const vector<int>& valid,
                  int sample_rate, int chunk, double speed, vector<VitJob>& pending)
{
  const size_t block_len = (mark_sync_frame_count() + mark_data_frame_count()) * Params::frame_size;
  auto queue = [&] (const vector<float>& soft, ConvBlockType code, double time, SyncFinder::Score score, ResultSet::Type type)
    {
      pending.push_back (VitJob { soft, code, time, score, type, key, chunk, speed });
    };
  vector<DecodedBlock> blocks;
  for (size_t i = 0; i < sync_scores.size(); i++)
    if (valid[i])
      {
        blocks.push_back ({ sync_scores[i].index, sync_scores[i].quality, sync_scores[i].block_type, &raw[i] });
        queue (raw[i], sync_scores[i].block_type, double (sync_scores[i].index) / sample_rate, sync_scores[i], ResultSet::Type::BLOCK);
      }
  /* ---- AB pairs */
  for (size_t i = 0; i < blocks.size(); i++)
    {
      if (blocks[i].type != ConvBlockType::b)
        continue;
      const int partner = nearest_block (blocks, 0, i, ConvBlockType::a, int (blocks[i].index) - int (block_len), Params::frame_size / 2);
      if (partner < 0)
        continue;
      const vector<float>& sa = *blocks[partner].soft, &sb = *blocks[i].soft;
      vector<float> interleaved (sa.size() * 2);
      for (size_t k = 0; k < sa.size(); k++)
        {
          interleaved[2 * k] = sa[k];
          interleaved[2 * k + 1] = sb[k];
        }
      queue (interleaved, ConvBlockType::ab, double (blocks[i].index) / sample_rate,
             SyncFinder::Score { blocks[i].index, (blocks[partner].quality + blocks[i].quality) / 2, ConvBlockType::ab }, ResultSet::Type::BLOCK);
    }
  /* ---- "all": the chain with the largest quality sum (the first one among equals) */
  vector<size_t> best;
  for (size_t head = 0; head < blocks.size(); head++)
    {
      const vector<size_t> chain = alternating_chain (blocks, head, block_len);
      if (chain_score (blocks, chain) > chain_score (blocks, best))
        best = chain;
    }
  if (best.size() > 1)
    {
      vector<float> mean_soft (code_size (ConvBlockType::ab, Params::payload_size));
      int members[2] = { 0, 0 };
      double quality_sum = 0;
      for (size_t b : best)
        {
          const int slot = blocks[b].type == ConvBlockType::b ? 1 : 0;
          const vector<float>& soft = *blocks[b].soft;
          for (size_t k = 0; k < soft.size(); k++)
            mean_soft[2 * k + slot] += soft[k];
          members[slot]++;
          quality_sum += blocks[b].quality;
        }
      for (size_t k = 0; k < mean_soft.size(); k++)
        mean_soft[k] /= max (members[k & 1], 1);
      queue (mean_soft, ConvBlockType::ab, 0.0, SyncFinder::Score { 0, quality_sum / (members[0] + members[1]), ConvBlockType::a }, ResultSet::Type::ALL);
    }
}

/* ---------------------------------------------------------------- BlockDecoder (src/wmget.cc:492-735) */

class BlockDecoder
{
  int debug_sync_frame_count = 0;
  const double speed;
  vector<SyncFinder::KeyResult> key_results;
public:
  explicit BlockDecoder (double speed) : speed (speed) {}

  /* the PCM (n_frames x n_channels at sample_rate) is already bound to the GPU context */
  void
  run (const vector<Key>& key_list, size_t n_frames, int n_channels, int sample_rate, vector<VitJob>& pending, int chunk)
  {
    SyncFinder sync_finder;
    key_results = sync_finder.search (key_list, n_frames, n_channels, SyncFinder::Mode::BLOCK, 0, n_frames * n_channels);
    for (const auto& key_result : key_results)
      {
        const Key& key = key_result.key;
        vector<uint64_t> indices;
        for (const auto& s : key_result.sync_scores)
          indices.push_back (s.index);
        vector<vector<float>> raw;
        vector<int> valid;
        if (!indices.empty() && !decode_raw_bits (key, indices, raw, valid))
          continue;
        build_block_jobs (key, key_result.sync_scores, raw, valid, sample_rate, chunk, speed, pending);
      }
    debug_sync_frame_count = n_frames / Params::frame_size;
  }
  string
  debug_sync()
  {
    if (key_results.size() != 1)
      return "";
    const auto& sync_scores = key_results[0].sync_scores;
    const int expect0 = Params::frames_pad_start * Params::frame_size;
    const int expect_step = (mark_sync_frame_count() + mark_data_frame_count()) * Params::frame_size;
    const int expect_end = debug_sync_frame_count * Params::frame_size;
    int sync_match = 0;
    for (int expect_index = expect0; expect_index + expect_step < expect_end; expect_index += expect_step)
      for (auto sync_score : sync_scores)
        if (abs (int (sync_score.index + Params::test_cut) - expect_index) < int (Params::frame_size / 2))
          {
            sync_match++;
            break;
          }
    return string_printf ("sync_match %d %zd\n", sync_match, sync_scores.size());
  }
};

/* ---------------------------------------------------------------- ClipDecoder (src/wmget.cc:737-884) */

class ClipDecoder
{
  const int frames_per_blk;
  const double speed;

  enum class Pos { START, END };
  void
  run_block (const vector<Key>& key_list, const float *samples, size_t n_frames, int n_channels, int sample_rate, vector<VitJob>& pending, int chunk, Pos pos)
  {
    awm_ctx *ctx = Engine::ctx();
    if (!ctx)
      return;
    const size_t n_values = n_frames * n_channels;
    const size_t n = size_t (frames_per_blk + 5) * Params::frame_size * n_channels;      // values of one padded block
    size_t first_sample, last_sample, pad_start = n, pad_end = n;
    if (pos == Pos::START)
      {
        first_sample = 0;
        last_sample = min (n, n_values);
        if (last_sample < n)                    // available samples + padding must always be one long block
          pad_start += n - last_sample;
      }
    else
      {
        if (n_values <= n)
          return;
        first_sample = n_values - n;
        last_sample = n_values;
      }
    const double time_offset = double (first_sample) / sample_rate / n_channels;
    /* scan_silence on the padded signal: [wav_first, wav_last) in value units */
    size_t nz_first = first_sample, nz_last = last_sample;
    while (nz_first < last_sample && samples[nz_first] == 0)
      nz_first++;
    while (nz_last > nz_first && samples[nz_last - 1] == 0)
      nz_last--;
    size_t wav_first, wav_last;
    const size_t ext_values = pad_start + (last_sample - first_sample) + pad_end;
    if (nz_first == last_sample)                // all zero
      wav_first = wav_last = ext_values;
    else
      {
        wav_first = pad_start + (nz_first - first_sample);
        wav_last = pad_start + (nz_last - first_sample);
      }
    const size_t ext_frames = ext_values / n_channels;
    if (awm_pcm_bind (ctx, samples + first_sample, (last_sample - first_sample) / n_channels, n_channels, pad_start / n_channels, pad_end / n_channels))
      {
        error ("audiowmark: %s\n", awm_last_error (ctx));
        return;
      }
    SyncFinder sync_finder;
    vector<SyncFinder::KeyResult> key_results = sync_finder.search (key_list, ext_frames, n_channels, SyncFinder::Mode::CLIP, wav_first, wav_last);
    const size_t count = mark_sync_frame_count() + mark_data_frame_count();
    for (const auto& key_result : key_results)
      {
        const Key& key = key_result.key;
        vector<uint64_t> indices;
        for (const auto& s : key_result.sync_scores)
          {
            indices.push_back (s.index);
            indices.push_back (s.index + count * Params::frame_size);
          }
        vector<vector<float>> raw;
        vector<int> valid;
        if (indices.empty() || !decode_raw_bits (key, indices, raw, valid))
          continue;
        for (size_t i = 0; i < key_result.sync_scores.size(); i++)
          if (valid[2 * i] && valid[2 * i + 1])
            {
              const auto& sync_score = key_result.sync_scores[i];
              const vector<float>& r1 = raw[2 * i], & r2 = raw[2 * i + 1];
              vector<float> raw_bit_vec (r1.size() * 2);
              for (size_t k = 0; k < r1.size(); k++)
                {
                  raw_bit_vec[2 * k]     = sync_score.block_type == ConvBlockType::a ? r1[k] : r2[k];
                  raw_bit_vec[2 * k + 1] = sync_score.block_type == ConvBlockType::a ? r2[k] : r1[k];
                }
              SyncFinder::Score sync_score_nopad = sync_score;
              sync_score_nopad.index = time_offset * sample_rate;
              pending.push_back (VitJob { raw_bit_vec, ConvBlockType::ab, time_offset, sync_score_nopad, ResultSet::Type::CLIP, key, chunk, speed });
            }
      }
  }
public:
  explicit ClipDecoder (double speed) : frames_per_blk (mark_sync_frame_count() + mark_data_frame_count()), speed (speed) {}
  bool wanted (size_t n_frames) const { return int (n_frames / Params::frame_size) < frames_per_blk * 3.1; }   /* clip decoder is only used for small inputs */
  void
  run (const vector<Key>& key_list, const float *samples, size_t n_frames, int n_channels, int sample_rate, vector<VitJob>& pending, int chunk)
  {
    const int wav_frames = n_frames / Params::frame_size;
    if (wav_frames < frames_per_blk * 3.1)       // clip decoder is only used for small inputs
      {
        run_block (key_list, samples, n_frames, n_channels, sample_rate, pending, chunk, Pos::START);
        run_block (key_list, samples, n_frames, n_channels, sample_rate, pending, chunk, Pos::END);
      }
  }
};

/* the audio of a chunk: float samples (host or device memory), or stored WAV sample bytes in host memory that are decoded on the
 * device (awm_pcm_bind_wav), so that only the stored bytes cross PCIe.  A whole 16 bit buffer lets the library find the overlap of
 * consecutive chunks inside it (awm_pcm_prefetch_s16); a streamed chunk marks it instead: its first `head` frames are the last ones
 * of the chunk before, already on the device, and `wav` holds only the frames after them. */
struct PcmRef
{
  const float   *f32 = nullptr;
  const void    *wav = nullptr;
  awm_wav_format fmt { 16, 0 };
  bool           streamed = false;
  size_t         head = 0;
  PcmRef advanced (size_t values) const       /* whole buffers only */
  {
    PcmRef r = *this;
    r.f32 = f32 ? f32 + values : nullptr;
    r.wav = wav ? static_cast<const unsigned char *> (wav) + values * (fmt.bits / 8) : nullptr;
    return r;
  }
  /* a streamed chunk with a head is bound once, from its prefetch; only the first chunk (no head) is bound again (decode_chunk) */
  int bind (awm_ctx *ctx, size_t n_frames, int n_channels) const
  {
    return f32 ? awm_pcm_bind (ctx, f32, n_frames, n_channels, 0, 0) : awm_pcm_bind_wav (ctx, wav, fmt, n_frames, n_channels, 0, 0);
  }
  int prefetch (awm_ctx *ctx, size_t n_frames, int n_channels) const
  {
    if (f32)
      return awm_pcm_prefetch (ctx, f32, n_frames, n_channels);
    if (streamed)
      return awm_pcm_prefetch_wav (ctx, wav, fmt, n_frames, n_channels, head);
    return awm_pcm_prefetch_s16 (ctx, static_cast<const int16_t *> (wav), n_frames, n_channels);
  }
  /* float samples in host memory (what the clip decoder cuts and pads): only needed for short inputs.  Called while this chunk is
   * the bound PCM: decoded WAV samples come from that device copy. */
  const float *host_floats (awm_ctx *ctx, size_t n_values, vector<float>& storage) const
  {
    const float *src = f32 ? f32 : awm_pcm_device (ctx, nullptr, nullptr);
    if (!src)
      return nullptr;
    if (f32 && !Engine::is_device_pointer (f32))
      return f32;
    storage.resize (n_values);
    if (awm_copy_to_host (ctx, storage.data(), src, n_values * sizeof (float)))
      return nullptr;
    return storage.data();
  }
};

/* decode (src/wmget.cc:886-939) for one chunk: everything up to the soft bits; the Viterbi jobs are queued */
int
decode_chunk (vector<VitJob>& pending, int chunk, string& debug_sync, const vector<Key>& key_list, const PcmRef& pcm, size_t n_frames,
              int n_channels, int sample_rate, bool first_chunk, bool print_speed_results = false)
{
  awm_ctx *ctx = Engine::ctx();
  if (!ctx)
    return 1;
  if (pcm.bind (ctx, n_frames, n_channels))
    {
      error ("audiowmark: %s\n", awm_last_error (ctx));
      return 1;
    }
  vector<float> host_storage;
  const float *host_samples = nullptr;          /* fetched lazily: only the clip decoder needs it */
  auto need_host = [&] () -> const float *
    {
      if (!host_samples)
        host_samples = pcm.host_floats (ctx, n_frames * n_channels, host_storage);
      return host_samples;
    };
  /* The strategy for integrating speed detection into decoding (src/wmget.cc:888-928):
   *  - the watermark is always decoded on the original data
   *  - if the detected speed is somewhat different from 1.0, stretched data is decoded as well
   *  - all normal and speed results are reported (the detected speed may be wrong on short clips) */
  if (Params::detect_speed || Params::detect_speed_patient || Params::try_speed > 0)
    {
      vector<DetectSpeedResult> speed_results;
      if (Params::detect_speed || Params::detect_speed_patient)
        {
          /* WAV samples: the float copy that was just bound on the device serves the speed scan as well */
          const float *speed_samples = pcm.f32 ? pcm.f32 : awm_pcm_device (ctx, nullptr, nullptr);
          speed_results = detect_speed (key_list, speed_samples, n_frames, n_channels, sample_rate, print_speed_results);
        }
      else
        for (const auto& key : key_list)
          speed_results.push_back ({ key, Params::try_speed });
      bool rebind = false;
      for (const auto& speed_result : speed_results)
        {
          /* resample_ratio (wav_data, speed, mark_sample_rate * speed): the stretched chunk stays on the device */
          const size_t speed_frames = lrint (double (n_frames) * speed_result.speed);
          const int speed_rate = Params::mark_sample_rate * speed_result.speed;
          if (rebind && pcm.bind (ctx, n_frames, n_channels))
            return 1;
          rebind = false;
          if (awm_pcm_push_resampled (ctx, speed_result.speed, 16, speed_frames))
            {
              error ("audiowmark: %s\n", awm_last_error (ctx));
              return 1;
            }
          BlockDecoder speed_block_decoder (speed_result.speed);
          speed_block_decoder.run ({ speed_result.key }, speed_frames, n_channels, speed_rate, pending, chunk);
          awm_pcm_pop (ctx);
          if (first_chunk && int (speed_frames / Params::frame_size) < (mark_sync_frame_count() + mark_data_frame_count()) * 3.1)
            {
              /* the clip decoder cuts and pads on the host: short inputs only, so the extra copy is small */
              vector<float> stretched;
              if (!need_host() || !resample_ratio (need_host(), n_frames, n_channels, speed_result.speed, stretched))
                return 1;
              ClipDecoder speed_clip_decoder (speed_result.speed);
              speed_clip_decoder.run ({ speed_result.key }, stretched.data(), speed_frames, n_channels, speed_rate, pending, chunk);
              rebind = true;
            }
        }
      if (rebind && pcm.bind (ctx, n_frames, n_channels))
        return 1;
    }
  const double tb0 = get_time();
  BlockDecoder block_decoder (1);
  block_decoder.run (key_list, n_frames, n_channels, sample_rate, pending, chunk);
  if (getenv ("AWM_TRACE"))
    fprintf (stderr, "[trace] chunk %d: block decoder (sync + soft bits) %.3f ms\n", chunk, (get_time() - tb0) * 1e3);
  if (first_chunk)
    {
      ClipDecoder clip_decoder (1);
      if (clip_decoder.wanted (n_frames))
        {
          if (!need_host())
            return 1;
          clip_decoder.run (key_list, need_host(), n_frames, n_channels, sample_rate, pending, chunk);
        }
    }
  debug_sync = block_decoder.debug_sync();
  return 0;
}

} // namespace get_detail

using namespace get_detail;

/* BlockDecoder job list of one chunk as flat records (for the multi-GPU driver):
 * u8 code_type (AWM_BLOCK_*), u8 pattern_type (ResultSet::Type), u8 score_block_type, u8 pad, f64 time, u64 index, f64 quality, u32 n_soft, f32 soft[] */
std::vector<unsigned char>
block_jobs_blob (const Key& key, const vector<SyncFinder::Score>& sync_scores, const vector<vector<float>>& raw, const vector<int>& valid, int sample_rate, int *n_jobs)
{
  vector<VitJob> jobs;
  build_block_jobs (key, sync_scores, raw, valid, sample_rate, 0, 1, jobs);
  std::vector<unsigned char> b;
  auto put = [&] (const void *p, size_t n) { const unsigned char *c = static_cast<const unsigned char *> (p); b.insert (b.end(), c, c + n); };
  for (const auto& j : jobs)
    {
      const uint8_t hdr[4] = { uint8_t (j.block_type == ConvBlockType::a ? AWM_BLOCK_A : j.block_type == ConvBlockType::b ? AWM_BLOCK_B : AWM_BLOCK_AB),
                               uint8_t (j.type), uint8_t (j.score.block_type), 0 };
      const double time = j.time, quality = j.score.quality;
      const uint64_t index = j.score.index;
      const uint32_t n_soft = j.soft.size();
      put (hdr, 4); put (&time, 8); put (&index, 8); put (&quality, 8); put (&n_soft, 4);
      put (j.soft.data(), n_soft * sizeof (float));
    }
  *n_jobs = int (jobs.size());
  return b;
}

/* chunk geometry of WavChunkLoader (src/wavchunkloader.cc:54-163): chunks of get_chunk_size minutes that
 * overlap by two blocks * 1.3 */
void
chunk_geometry (int sample_rate, size_t& max_frames, size_t& overlap_frames)
{
  max_frames = lrint (Params::get_chunk_size * 60 * sample_rate);
  const double block_seconds = (mark_sync_frame_count() + mark_data_frame_count()) * Params::frame_size / double (Params::mark_sample_rate);
  overlap_frames = lrint (2 * block_seconds * 1.3 * sample_rate);
}

int
get_watermark_buffer (const vector<Key>& key_list, const float *samples, size_t n_frames, int n_channels, int sample_rate, ResultSet& result_set,
                      bool print_speed_results, size_t *mark_rate_frames)
{
  return get_watermark_pcm (key_list, samples, nullptr, n_frames, n_channels, sample_rate, result_set, print_speed_results, mark_rate_frames);
}

int
get_watermark_buffer_s16 (const vector<Key>& key_list, const int16_t *samples, size_t n_frames, int n_channels, int sample_rate, ResultSet& result_set,
                          bool print_speed_results, size_t *mark_rate_frames)
{
  return get_watermark_pcm (key_list, nullptr, samples, n_frames, n_channels, sample_rate, result_set, print_speed_results, mark_rate_frames);
}

static int merge_chunks (vector<VitJob>& pending, const vector<double>& time_offsets, const vector<string>& debug_syncs, const vector<Key>& key_list,
                         ResultSet& result_set);

int
get_watermark_pcm (const vector<Key>& key_list, const float *samples, const int16_t *samples16, size_t n_frames, int n_channels, int sample_rate,
                   ResultSet& result_set, bool print_speed_results, size_t *mark_rate_frames)
{
  vector<float> resampled, converted;
  if (samples16 && sample_rate != Params::mark_sample_rate)
    {
      /* rare combination: convert on the host, then take the float path through the resampler */
      converted.resize (n_frames * n_channels);
      const float norm = 1.0 / 0x80000000LL;
      for (size_t i = 0; i < converted.size(); i++)
        converted[i] = (int (samples16[i]) << 16) * norm;
      samples = converted.data();
      samples16 = nullptr;
    }
  if (sample_rate != Params::mark_sample_rate)
    {
      /* WavChunkLoader resamples the input to the watermark rate while it reads (src/wavchunkloader.cc:66-73, 196-221) */
      const double ratio = double (Params::mark_sample_rate) / sample_rate;
      awm_ctx *rctx = Engine::ctx();
      if (!rctx)
        return 1;
      const size_t n_out = resample_stream_frames (n_frames, ratio);
      resampled.assign (n_out * n_channels, 0.f);
      if (awm_resample (rctx, samples, n_frames, n_channels, ratio, 16, resampled.data(), n_out))
        {
          error ("audiowmark: %s\n", awm_last_error (rctx));
          return 1;
        }
      samples = resampled.data();
      samples16 = nullptr;
      n_frames = n_out;
      sample_rate = Params::mark_sample_rate;
    }
  if (mark_rate_frames)
    *mark_rate_frames = n_frames;
  size_t max_frames, overlap;
  chunk_geometry (sample_rate, max_frames, overlap);
  size_t start = 0, end = min (max_frames, n_frames);
  double time_offset = 0;
  bool first_chunk = true, eof = end < max_frames;
  if (n_frames == 0)
    return 0;
  /* pass 1: sync search + soft bits per chunk (GPU), Viterbi jobs of all chunks are collected */
  vector<VitJob> pending;
  vector<double> time_offsets;
  vector<string> debug_syncs;
  awm_ctx *ctx = Engine::ctx();
  if (!ctx)
    return 1;
  /* host buffers: the next chunk travels over PCIe while the current one is searched */
  PcmRef pcm;
  pcm.f32 = samples16 ? nullptr : samples;
  pcm.wav = samples16;
  pcm.prefetch (ctx, end - start, n_channels);
  for (;;)
    {
      string debug_sync;
      if (!eof)
        {
          const size_t nstart = end - overlap, nend = min (nstart + max_frames, n_frames);
          pcm.advanced (nstart * n_channels).prefetch (ctx, nend - nstart, n_channels);
        }
      if (decode_chunk (pending, int (time_offsets.size()), debug_sync, key_list, pcm.advanced (start * n_channels), end - start, n_channels, sample_rate, first_chunk, print_speed_results))
        return 1;
      time_offsets.push_back (time_offset);
      debug_syncs.push_back (debug_sync);
      first_chunk = false;
      if (eof)
        break;
      time_offset += double (end - start - overlap) / sample_rate;
      start = end - overlap;
      const size_t new_end = min (start + max_frames, n_frames);
      eof = (new_end - start) < max_frames;
      end = new_end;
    }
  return merge_chunks (pending, time_offsets, debug_syncs, key_list, result_set);
}

/* pass 2 of a chunk loop: one Viterbi launch for the code words of all chunks, then the reference's per-chunk merge in chunk order */
static int
merge_chunks (vector<VitJob>& pending, const vector<double>& time_offsets, const vector<string>& debug_syncs, const vector<Key>& key_list,
              ResultSet& result_set)
{
  vector<ResultSet> chunk_results (time_offsets.size());
  const double tv0 = get_time();
  const size_t n_jobs = pending.size();
  if (!run_viterbi_jobs (pending, chunk_results))
    return 1;
  if (getenv ("AWM_TRACE"))
    fprintf (stderr, "[trace] viterbi: %zu jobs %.3f ms\n", n_jobs, (get_time() - tv0) * 1e3);
  for (size_t c = 0; c < chunk_results.size(); c++)
    {
      chunk_results[c].set_debug_sync (debug_syncs[c]);
      chunk_results[c].apply_time_offset (time_offsets[c]);
      result_set.merge (chunk_results[c]);
    }
  result_set.sort (key_list);
  return 0;
}

/* ---------------------------------------------------------------- streamed input (WavChunkLoader, src/wavchunkloader.cc:54-163) */

namespace {

/* Reads the chunks of one input on a thread of its own into two page-locked buffers of stored sample bytes, chunk k into buffer
 * k % 2: the next chunk is read while the current one is searched, and host memory stays at two chunks whatever the input length.
 * Chunk 0 asks for first_frames frames, every later chunk for next_frames (the frames after its overlap, which is on the device
 * already), never more than limit_frames in all.  A chunk that gets fewer frames than it asked for is the last; the thread stops
 * there, on a read error, or when the reader is destroyed, and the destructor joins it on every path.  The source is read
 * piece_frames frames at a time (0: a whole chunk per call), so that stopping never waits for more than one piece. */
class ChunkReader
{
public:
  using Source = std::function<Error (unsigned char *dst, size_t count, size_t *n_read)>;

  ChunkReader (Source source, size_t frame_bytes, size_t first_frames, size_t next_frames, size_t limit_frames, size_t piece_frames) :
    m_source (source), m_frame_bytes (frame_bytes), m_first (first_frames), m_next (next_frames), m_limit (limit_frames),
    m_piece (piece_frames ? piece_frames : std::max (first_frames, size_t (1)))
  {
    /* buffer 1 holds chunks 1, 3, ...: not needed when the whole input fits into chunk 0 */
    const size_t frames[2] = { min (m_first, m_limit), m_limit > m_first ? m_next : 0 };
    for (int b = 0; b < 2; b++)
      {
        const size_t bytes = std::max<size_t> (frames[b] * m_frame_bytes, 1);
        m_slot[b].data = static_cast<unsigned char *> (awm_host_alloc (bytes));
        m_slot[b].pinned = m_slot[b].data != nullptr;
        if (!m_slot[b].data)                    /* pageable memory works too, the copies are only slower */
          m_slot[b].data = static_cast<unsigned char *> (malloc (bytes));
        if (!m_slot[b].data)
          return;
      }
    m_thread = std::thread ([this] { run(); });
  }
  ~ChunkReader()
  {
    {
      std::lock_guard<std::mutex> lock (m_mutex);
      m_stop = true;
    }
    m_cond.notify_all();
    if (m_thread.joinable())
      m_thread.join();
    for (Slot& s : m_slot)
      if (s.data)
        s.pinned ? awm_host_free (s.data) : free (s.data);
  }
  bool ok() const { return m_thread.joinable(); }

  /* waits until chunk k has been read: its bytes and frame count, or the read error */
  Error
  take (int k, const unsigned char **bytes, size_t *n_frames)
  {
    Slot& s = m_slot[k & 1];
    std::unique_lock<std::mutex> lock (m_mutex);
    m_cond.wait (lock, [&] { return s.state == Slot::READY; });
    *bytes = s.data;
    *n_frames = s.n_frames;
    return s.error;
  }
  /* the bytes of chunk k have reached the device: its buffer may take chunk k + 2 */
  void
  release (int k)
  {
    {
      std::lock_guard<std::mutex> lock (m_mutex);
      m_slot[k & 1].state = Slot::FREE;
    }
    m_cond.notify_all();
  }

private:
  struct Slot
  {
    enum State { FREE, FILLING, READY } state = FREE;
    unsigned char *data = nullptr;
    bool   pinned = false;
    size_t n_frames = 0;
    Error  error;
  };
  Source                  m_source;
  const size_t            m_frame_bytes, m_first, m_next, m_limit, m_piece;
  Slot                    m_slot[2];
  std::mutex              m_mutex;
  std::condition_variable m_cond;
  std::atomic<bool>       m_stop { false };
  std::thread             m_thread;

  void
  run()
  {
    size_t total = 0;
    for (int k = 0;; k++)
      {
        Slot& s = m_slot[k & 1];
        {
          std::unique_lock<std::mutex> lock (m_mutex);
          m_cond.wait (lock, [&] { return m_stop || s.state == Slot::FREE; });
          if (m_stop)
            return;
          s.state = Slot::FILLING;
        }
        const size_t ask = k ? m_next : m_first, want = min (ask, m_limit - total);
        size_t got = 0;
        Error err;
        while (got < want && !m_stop)
          {
            size_t n = 0;
            err = m_source (s.data + got * m_frame_bytes, min (m_piece, want - got), &n);
            if (err || !n)
              break;
            got += n;
          }
        total += got;
        {
          std::lock_guard<std::mutex> lock (m_mutex);
          s.n_frames = got;
          s.error = err;
          s.state = Slot::READY;
        }
        m_cond.notify_all();
        if (err || got < ask || m_stop)
          return;
      }
  }
};

} // namespace

/* `get` on a stream of stored WAV samples at the watermark rate, chunk by chunk with WavChunkLoader's geometry and EOF rule (an input
 * that is an exact multiple of the chunk size ends with a chunk that holds only the overlap): chunk k + 1 is read on the reader thread
 * while chunk k is searched, the overlap is taken from the device copy of the chunk before, and every byte of the input crosses PCIe
 * once, in its stored format.  n_frames_hint: the length if the stream knows it (sizes the host buffers), else N_FRAMES_UNKNOWN.
 * --test-truncate cuts the stream as it cut the loaded file.  A read error goes to read_error (the caller words the message). */
int
get_watermark_stream (const vector<Key>& key_list, const std::function<Error (unsigned char *, size_t, size_t *)>& source, awm_wav_format format,
                      int n_channels, size_t n_frames_hint, size_t piece_frames, ResultSet& result_set, bool print_speed_results,
                      size_t *n_frames_out, Error& read_error)
{
  const int sample_rate = Params::mark_sample_rate;
  size_t max_frames, overlap;
  chunk_geometry (sample_rate, max_frames, overlap);
  size_t limit = n_frames_hint;
  if (Params::test_truncate)
    limit = min (limit, size_t (sample_rate) * Params::test_truncate);
  *n_frames_out = 0;
  awm_ctx *ctx = Engine::ctx();
  if (!ctx)
    return 1;
  ChunkReader reader (source, size_t (format.bits / 8) * n_channels, max_frames, max_frames - overlap, limit, piece_frames);
  if (!reader.ok())
    {
      error ("audiowmark: out of memory for the input buffers\n");
      return 1;
    }
  /* pass 1: sync search + soft bits per chunk (GPU), Viterbi jobs of all chunks are collected */
  vector<VitJob> pending;
  vector<double> time_offsets;
  vector<string> debug_syncs;
  size_t chunk_frames = 0;
  double time_offset = 0;
  for (int k = 0;; k++)
    {
      const unsigned char *bytes;
      size_t n_new;
      read_error = reader.take (k, &bytes, &n_new);
      if (read_error)
        return 1;
      *n_frames_out += n_new;
      if (k == 0 && n_new == 0)                 /* empty input: no chunk at all */
        break;
      PcmRef pcm;
      pcm.wav = bytes;
      pcm.fmt = format;
      pcm.streamed = true;
      pcm.head = k ? overlap : 0;
      if (k)
        time_offset += double (chunk_frames - overlap) / sample_rate;
      chunk_frames = pcm.head + n_new;
      const bool eof = chunk_frames < max_frames;
      if (pcm.prefetch (ctx, chunk_frames, n_channels))
        {
          error ("audiowmark: %s\n", awm_last_error (ctx));
          return 1;
        }
      string debug_sync;
      if (decode_chunk (pending, k, debug_sync, key_list, pcm, chunk_frames, n_channels, sample_rate, k == 0, print_speed_results))
        return 1;
      time_offsets.push_back (time_offset);
      debug_syncs.push_back (debug_sync);
      if (eof)
        break;
      if (awm_synchronize (ctx))                /* the copy of this chunk's bytes has completed */
        {
          error ("audiowmark: %s\n", awm_last_error (ctx));
          return 1;
        }
      reader.release (k);
    }
  return merge_chunks (pending, time_offsets, debug_syncs, key_list, result_set);
}

int
get_watermark_chunk (const vector<Key>& key_list, const float *samples, size_t n_frames, int n_channels, int sample_rate,
                     bool first_chunk, ResultSet& chunk_result)
{
  if (sample_rate != Params::mark_sample_rate)
    {
      error ("audiowmark: input sample rate %d: only %d Hz is supported\n", sample_rate, Params::mark_sample_rate);
      return 1;
    }
  vector<VitJob> pending;
  string debug_sync;
  PcmRef pcm;
  pcm.f32 = samples;
  if (decode_chunk (pending, 0, debug_sync, key_list, pcm, n_frames, n_channels, sample_rate, first_chunk))
    return 1;
  vector<ResultSet> one (1);
  if (!run_viterbi_jobs (pending, one))
    return 1;
  one[0].set_debug_sync (debug_sync);
  chunk_result.merge (one[0]);
  return 0;
}

static int
report (ResultSet& result_set, size_t time_length, const vector<int>& orig_bits)
{
  if (!Params::json_output.empty())
    result_set.print_json (time_length, Params::json_output);
  if (Params::json_output != "-")
    result_set.print();
  if (!orig_bits.empty())
    {
      const int match_count = result_set.print_match_count (orig_bits);
      result_set.print_debug_sync();
      if (Params::expect_matches >= 0)
        {
          printf ("expect_matches %d\n", Params::expect_matches);
          if (match_count != Params::expect_matches)
            return 1;
        }
      else if (!match_count)
        return 1;
    }
  return 0;
}

int
get_watermark (const vector<Key>& key_list, const string& infile, const string& orig_pattern)
{
  vector<int> orig_bitvec;
  if (!orig_pattern.empty())
    {
      orig_bitvec = parse_payload (orig_pattern);
      if (orig_bitvec.empty())
        return 1;
    }
  Error err;
  std::unique_ptr<AudioInputStream> in_stream = AudioInputStream::create (infile, err);
  if (err)
    {
      error ("audiowmark: error loading %s: %s\n", infile.c_str(), err.message());
      return 1;
    }
  ResultSet result_set;
  size_t mark_rate_frames = 0;
  WavInputStream *wav_in = dynamic_cast<WavInputStream *> (in_stream.get());
  if (wav_in && wav_in->sample_rate() == Params::mark_sample_rate)
    {
      /* streamed: host memory stays at two chunks of stored bytes for any input length (WavChunkLoader) */
      const RawFormat& f = wav_in->raw_format();
      const awm_wav_format format { f.bit_depth(), f.encoding() == Encoding::FLOAT ? 1 : 0 };
      auto source = [wav_in] (unsigned char *dst, size_t count, size_t *n_read) { return wav_in->read_raw_frames (dst, count, n_read); };
      Error read_err;
      if (get_watermark_stream (key_list, source, format, f.n_channels(), wav_in->n_frames(), 65536, result_set, !orig_bitvec.empty(),
                                &mark_rate_frames, read_err))
        {
          if (read_err)
            error ("audiowmark: error loading %s: %s\n", infile.c_str(), read_err.message());
          return 1;
        }
    }
  else
    {
      /* other sample rates are resampled as a whole and then cut into chunks (a streaming resampler would first have to equal the
       * whole-buffer one bit for bit), and raw input is converted on the host: the whole input is loaded first */
      WavData wav;
      err = wav.load (in_stream.get());
      if (err)
        {
          error ("audiowmark: error loading %s: %s\n", infile.c_str(), err.message());
          return 1;
        }
      if (Params::test_truncate)
        {
          const size_t want = size_t (wav.sample_rate()) * wav.n_channels() * Params::test_truncate;
          if (want < wav.n_values())
            wav.mutable_samples().resize (want);
        }
      if (get_watermark_buffer (key_list, wav.samples().data(), wav.n_frames(), wav.n_channels(), wav.sample_rate(), result_set, !orig_bitvec.empty(),
                                &mark_rate_frames))
        return 1;
    }
  const size_t time_length = lrint (mark_rate_frames / double (Params::mark_sample_rate));
  return report (result_set, time_length, orig_bitvec);
}
