// awm_wm.hh -- entry points of the watermark drivers, same names / argument meaning as the reference
// (src/wmcommon.hh:226-228, src/syncfinder.hh:71-121).
#pragma once
#include <functional>
#include <string>
#include <vector>
#include "awm_params.hh"
#include "awm_random.hh"
#include "awm_code.hh"
#include "awm_streams.hh"
#include "../../include/awm_b200.h"

int add_stream_watermark (const Key& key, AudioInputStream *in_stream, AudioOutputStream *out_stream, const std::string& bits, size_t zero_frames);
int add_watermark (const Key& key, const std::string& infile, const std::string& outfile, const std::string& bits);
int get_watermark (const std::vector<Key>& key_list, const std::string& infile, const std::string& orig_pattern);

/* buffer-level drivers used by the C host API (bench / tests): same computation without file I/O */
struct AddStats { int data_blocks = 0; double snr_db = 0; };
int add_watermark_buffer (const Key& key, const float *in, float *out, size_t n_frames, int n_channels, int sample_rate,
                          const std::string& bits, AddStats *stats, uint64_t first_frame_number = 0);

/* add_stream_watermark's loop with bounded memory (window by window; see awm_add.cc); callbacks read / write interleaved frames */
int add_watermark_windowed (const Key& key, const std::function<Error (std::vector<float>&, size_t)>& read,
                            const std::function<Error (const std::vector<float>&)>& write, int n_channels, int sample_rate, const std::string& bits,
                            size_t zero_frames, size_t window_frames, AddStats *stats, size_t *frames_written);

/* frame counts of the add loop for inputs that are not at the watermark rate (see awm_add.cc) */
void resampled_add_plan (size_t n_frames, int sample_rate, bool limiter_on, size_t limiter_block, size_t& n_emit, size_t& gen_runs_out);

class ResultSet;
int get_watermark_buffer (const std::vector<Key>& key_list, const float *samples, size_t n_frames, int n_channels, int sample_rate,
                          ResultSet& result_set, bool print_speed_results = false, size_t *mark_rate_frames = nullptr);

/* 16 bit PCM in host memory (what a 16 bit WAV file holds): converted on the device, identical results at half the PCIe traffic */
int get_watermark_buffer_s16 (const std::vector<Key>& key_list, const int16_t *samples, size_t n_frames, int n_channels, int sample_rate,
                              ResultSet& result_set, bool print_speed_results = false, size_t *mark_rate_frames = nullptr);
int get_watermark_pcm (const std::vector<Key>& key_list, const float *samples, const int16_t *samples16, size_t n_frames, int n_channels, int sample_rate,
                       ResultSet& result_set, bool print_speed_results, size_t *mark_rate_frames);
int add_watermark_buffer_s16 (const Key& key, const int16_t *in, int16_t *out, size_t n_frames, int n_channels, int sample_rate,
                              const std::string& bits, AddStats *stats, uint64_t first_frame_number = 0);

/* `get` on a stream of stored WAV samples at mark_sample_rate, read chunk by chunk (WavChunkLoader): source (dst, count, &n_read)
 * delivers the bytes of up to count frames, n_read = 0 at the end.  The CLI reads a WavInputStream, awmh_get_wav a memory buffer. */
int get_watermark_stream (const std::vector<Key>& key_list, const std::function<Error (unsigned char *, size_t, size_t *)>& source,
                          awm_wav_format format, int n_channels, size_t n_frames_hint, size_t piece_frames, ResultSet& result_set,
                          bool print_speed_results, size_t *n_frames_out, Error& read_error);

/* chunk-level pieces of get_watermark_buffer for sharded runs (one process per GPU): a rank decodes some of the
 * reference's chunks (WavChunkLoader geometry) and the chunk result sets are merged in chunk order afterwards */
int get_watermark_chunk (const std::vector<Key>& key_list, const float *samples, size_t n_frames, int n_channels, int sample_rate,
                         bool first_chunk, ResultSet& chunk_result);
void chunk_geometry (int sample_rate, size_t& max_frames, size_t& overlap_frames);

int frame_count (const WavData& wav_data);

class SyncFinder
{
public:
  enum class Mode { BLOCK, CLIP };
  struct Score { size_t index; double quality; ConvBlockType block_type; };
  struct KeyResult { Key key; std::vector<Score> sync_scores; };
  /* searches the PCM currently bound to the GPU context; n_frames/n_channels describe it
   * (padded length for CLIP mode), wav_first/wav_last = non-silent value range */
  std::vector<KeyResult> search (const std::vector<Key>& key_list, size_t n_frames, int n_channels, Mode mode,
                                 size_t wav_first, size_t wav_last);
  static double normalize_sync_quality (double raw_quality);

  /* test aid: when tracing is on every search() call appends what it returns (mode, length of the searched signal and per key
   * the final scores), so that tests can compare sync positions exactly with the reference's SyncFinder::search */
  struct TraceRecord { Mode mode; size_t n_frames; std::vector<Score> scores; };
  static void trace_enable (bool on);
  static std::vector<TraceRecord> trace_take();
};

/* stage functions of SyncFinder::search / BlockDecoder::run, used by get_watermark_buffer and by the frame-balanced
 * multi-GPU driver (audiowmark_b200/sharding.py), which runs the GPU stages on slices of a chunk on different ranks */
int  select_candidates_from_peaks (const awm_search_score *peaks, size_t n, double floor_q, double threshold, std::vector<awm_search_score>& out);
void select_final_scores (std::vector<awm_search_score>& scores, std::vector<SyncFinder::Score>& out);

