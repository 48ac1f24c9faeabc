// awm_streams.hh -- the stream / WavData surface of the host side.
// Same abstract interface as the reference (src/audiostream.hh:31-62, src/wavdata.hh:27-74,
// src/rawinputstream.hh:28-56, src/rawconverter.hh:23-50): read_frames() fills at most `count`
// sample-frames of interleaved floats and returns an EMPTY vector at EOF; Error is truthy on failure.
// Implementations here are dependency free: RIFF/RF64 WAV (PCM 8/16/24/32, float 32/64,
// WAVE_FORMAT_EXTENSIBLE), wav-pipe, headerless raw.  No libsndfile / mpg123.
#pragma once
#include <memory>
#include <stdio.h>
#include <string>
#include <vector>
#include "awm_util.hh"

enum class Encoding { SIGNED, UNSIGNED, FLOAT };

class AudioStream
{
public:
  virtual int bit_depth()   const = 0;
  virtual int sample_rate() const = 0;
  virtual int n_channels()  const = 0;
  virtual ~AudioStream() {}
};

class AudioInputStream : public AudioStream
{
public:
  static std::unique_ptr<AudioInputStream> create (const std::string& filename, Error& err);
  static constexpr size_t N_FRAMES_UNKNOWN = ~size_t (0);
  virtual size_t   n_frames() const = 0;
  virtual Encoding encoding() const = 0;
  virtual Error    read_frames (std::vector<float>& samples, size_t count) = 0;
};

class AudioOutputStream : public AudioStream
{
public:
  static std::unique_ptr<AudioOutputStream> create (const std::string& filename, int n_channels, int sample_rate,
                                                    int bit_depth, Encoding encoding, size_t n_frames, Error& err);
  virtual Error write_frames (const std::vector<float>& frames) = 0;
  virtual Error close() = 0;
};

class RawFormat
{
public:
  enum Endian { LITTLE, BIG };
private:
  int      m_n_channels  = 2;
  int      m_sample_rate = 0;
  int      m_bit_depth   = 16;
  Endian   m_endian      = LITTLE;
  Encoding m_encoding    = Encoding::SIGNED;
public:
  RawFormat() {}
  RawFormat (int n_channels, int sample_rate, int bit_depth) : m_n_channels (n_channels), m_sample_rate (sample_rate), m_bit_depth (bit_depth) {}
  int      n_channels() const  { return m_n_channels; }
  int      sample_rate() const { return m_sample_rate; }
  int      bit_depth() const   { return m_bit_depth; }
  Endian   endian() const      { return m_endian; }
  Encoding encoding() const    { return m_encoding; }
  void set_channels (int c)        { m_n_channels = c; }
  void set_sample_rate (int r)     { m_sample_rate = r; }
  void set_bit_depth (int b)       { m_bit_depth = b; }
  void set_endian (Endian e)       { m_endian = e; }
  void set_encoding (Encoding e)   { m_encoding = e; }
};

/* float <-> PCM with the reference's rounding rules (src/rawconverter.hh:34-64, src/rawconverter.cc:155-286) */
template<int BITS> static inline int
float_to_int_clip (float f)
{
  const int64_t inorm = (1LL << (BITS - 1));
  const float   snorm = f * float (inorm);
  if (snorm >= float (inorm - 1))
    return inorm - 1;
  if (snorm <= float (-inorm))
    return -inorm;
  return int (snorm);       // truncates toward zero
}
static inline float
float_clip (float f)
{
  return f >= 1.f ? 1.f : (f <= -1.f ? -1.f : f);
}

class RawConverter
{
  RawFormat m_format;
public:
  static RawConverter *create (const RawFormat& raw_format, Error& error);
  explicit RawConverter (const RawFormat& f) : m_format (f) {}
  void to_raw   (const float *samples, unsigned char *bytes, size_t n_samples) const;
  void from_raw (const unsigned char *bytes, float *samples, size_t n_samples) const;
};

class RawInputStream : public AudioInputStream
{
  RawFormat m_format;
  FILE     *m_file = nullptr;
  bool      m_close = false;
  std::unique_ptr<RawConverter> m_conv;
  std::vector<unsigned char> m_bytes;
public:
  ~RawInputStream();
  Error    open (const std::string& filename, const RawFormat& format);
  Error    read_frames (std::vector<float>& samples, size_t count) override;
  int      bit_depth() const override   { return m_format.bit_depth(); }
  int      sample_rate() const override { return m_format.sample_rate(); }
  int      n_channels() const override  { return m_format.n_channels(); }
  size_t   n_frames() const override    { return N_FRAMES_UNKNOWN; }
  Encoding encoding() const override    { return m_format.encoding(); }
};

class RawOutputStream : public AudioOutputStream
{
  RawFormat m_format;
  FILE     *m_file = nullptr;
  bool      m_close = false;
  std::unique_ptr<RawConverter> m_conv;
public:
  ~RawOutputStream();
  Error open (const std::string& filename, const RawFormat& format);
  Error write_frames (const std::vector<float>& frames) override;
  Error close() override;
  int   bit_depth() const override   { return m_format.bit_depth(); }
  int   sample_rate() const override { return m_format.sample_rate(); }
  int   n_channels() const override  { return m_format.n_channels(); }
};

/* RIFF / RF64 reader.  pipe_mode = true is the reference's WavPipeInputStream (src/wavpipeinputstream.cc:69-173):
 * length unknown, samples are read until EOF.  pipe_mode = false stands in for the libsndfile reader
 * (src/sfinputstream.cc): the data chunk size bounds the stream and n_frames() is known. */
class WavInputStream : public AudioInputStream
{
  RawFormat m_format;
  FILE     *m_file = nullptr;
  bool      m_close = false;
  bool      m_pipe_mode = false;
  size_t    m_n_frames = N_FRAMES_UNKNOWN;
  size_t    m_frames_left = 0;
  std::unique_ptr<RawConverter> m_conv;
  std::vector<unsigned char> m_bytes;
public:
  ~WavInputStream();
  Error    open (const std::string& filename, bool pipe_mode);
  Error    read_frames (std::vector<float>& samples, size_t count) override;
  /* the undecoded sample bytes of up to `count` frames (what read_frames would convert) into bytes[0 .. count * frame size);
   * *n_read = frames delivered, 0 at EOF.  *format (if given) = how the bytes are stored: bit depth, encoding (8 bit is UNSIGNED,
   * float WAVs FLOAT, everything else SIGNED), little endian, channels, sample rate. */
  Error    read_raw_frames (unsigned char *bytes, size_t count, size_t *n_read, RawFormat *format = nullptr);
  const RawFormat& raw_format() const   { return m_format; }
  int      bit_depth() const override   { return m_format.bit_depth(); }
  int      sample_rate() const override { return m_format.sample_rate(); }
  int      n_channels() const override  { return m_format.n_channels(); }
  size_t   n_frames() const override    { return m_n_frames; }
  Encoding encoding() const override    { return m_format.encoding() == Encoding::UNSIGNED && !m_pipe_mode ? Encoding::SIGNED : m_format.encoding(); }
};

/* WAV writer: to a file (stand-in for the libsndfile writer, src/sfoutputstream.cc: integer samples are
 * float_to_int_clip<32> and the file keeps the most significant bits) or to stdout
 * (src/stdoutwavoutputstream.cc:75-191: RawConverter rounding, optional wav-pipe header with size -1). */
class WavOutputStream : public AudioOutputStream
{
  FILE    *m_file = nullptr;
  bool     m_close = false;
  bool     m_to_stdout = false, m_rf64 = false, m_float = false;
  int      m_bit_depth = 0, m_sample_rate = 0, m_n_channels = 0;
  uint64_t m_data_bytes = 0;
  bool     m_open = false;
  std::unique_ptr<RawConverter> m_conv;
  void     write_header (uint64_t data_bytes, bool wav_pipe);
public:
  ~WavOutputStream();
  Error open_file (const std::string& filename, int n_channels, int sample_rate, int bit_depth, Encoding encoding, bool rf64);
  Error open_stdout (int n_channels, int sample_rate, int bit_depth, Encoding encoding, size_t n_frames, bool wav_pipe);
  Error write_frames (const std::vector<float>& frames) override;
  Error close() override;
  int   bit_depth() const override   { return m_bit_depth; }
  int   sample_rate() const override { return m_sample_rate; }
  int   n_channels() const override  { return m_n_channels; }
};

class WavData
{
  std::vector<float> m_samples;
  int m_n_channels = 0, m_sample_rate = 0, m_bit_depth = 0;
public:
  WavData() {}
  WavData (const std::vector<float>& samples, int n_channels, int sample_rate, int bit_depth) :
    m_samples (samples), m_n_channels (n_channels), m_sample_rate (sample_rate), m_bit_depth (bit_depth) {}
  Error load (AudioInputStream *in_stream);
  Error load (const std::string& filename);
  Error save (const std::string& filename) const;
  int    sample_rate() const { return m_sample_rate; }
  int    bit_depth() const   { return m_bit_depth; }
  int    n_channels() const  { return m_n_channels; }
  size_t n_values() const    { return m_samples.size(); }
  size_t n_frames() const    { return m_n_channels ? m_samples.size() / m_n_channels : 0; }
  const std::vector<float>& samples() const { return m_samples; }
  std::vector<float>& mutable_samples()     { return m_samples; }
  void set_samples (const std::vector<float>& samples) { m_samples = samples; }
};
