#include "awm_streams.hh"
#include "awm_params.hh"

#include <errno.h>
#include <string.h>
#include <algorithm>

using std::string;
using std::vector;

/* ---------------------------------------------------------------- RawConverter */

/* 16 bit little-endian signed PCM is what nearly every file holds: straight loops the compiler vectorises (the generic code below
 * assembles every sample byte by byte).  Same arithmetic: reading = sample * 2^-15, writing = the rule passed in. */
__attribute__ ((optimize ("O3"))) static void
s16le_to_float (const unsigned char *bytes, float *samples, size_t n)
{
  for (size_t i = 0; i < n; i++)
    {
      int16_t v;
      memcpy (&v, bytes + 2 * i, 2);
      samples[i] = float (v) * (1.0f / 32768.0f);           // exact, == (v << 16) * 2^-31
    }
}

/* float_to_int_clip<32> (f) >> 16 (libsndfile's int API keeps the most significant bits) */
__attribute__ ((optimize ("O3"))) static void
float_to_s16le_msb (const float *samples, unsigned char *bytes, size_t n)
{
  for (size_t i = 0; i < n; i++)
    {
      const float sn = samples[i] * 2147483648.0f;
      const int32_t v = sn >= 2147483648.0f ? INT32_MAX : (sn <= -2147483648.0f ? INT32_MIN : int32_t (sn));
      const int16_t w = int16_t (v >> 16);
      memcpy (bytes + 2 * i, &w, 2);
    }
}

/* float_to_int_clip<16> (f): rounding at 16 bit (RawConverter, stdout / raw streams) */
__attribute__ ((optimize ("O3"))) static void
float_to_s16le_clip16 (const float *samples, unsigned char *bytes, size_t n)
{
  for (size_t i = 0; i < n; i++)
    {
      const float sn = samples[i] * 32768.0f;
      const int32_t v = sn >= 32767.0f ? 32767 : (sn <= -32768.0f ? -32768 : int32_t (sn));
      const int16_t w = int16_t (v);
      memcpy (bytes + 2 * i, &w, 2);
    }
}

RawConverter *
RawConverter::create (const RawFormat& f, Error& error)
{
  error = Error::Code::NONE;
  if (f.encoding() == Encoding::FLOAT)
    {
      if (f.bit_depth() != 32 && f.bit_depth() != 64)
        {
          error = Error (string_printf ("unsupported bit depth %d for float encoding", f.bit_depth()));
          return nullptr;
        }
    }
  else if (f.bit_depth() != 8 && f.bit_depth() != 16 && f.bit_depth() != 24 && f.bit_depth() != 32)
    {
      error = Error (string_printf ("unsupported bit depth %d for signed/unsigned encoding", f.bit_depth()));
      return nullptr;
    }
  return new RawConverter (f);
}

void
RawConverter::to_raw (const float *samples, unsigned char *bytes, size_t n) const
{
  const int width = m_format.bit_depth() / 8;
  const bool little = m_format.endian() == RawFormat::LITTLE;
  if (m_format.encoding() == Encoding::FLOAT)
    {
      for (size_t i = 0; i < n; i++, bytes += width)
        {
          unsigned char tmp[8];
          if (width == 4)
            {
              const float f = float_clip (samples[i]);
              memcpy (tmp, &f, 4);
            }
          else
            {
              const double d = float_clip (samples[i]);
              memcpy (tmp, &d, 8);
            }
          for (int b = 0; b < width; b++)         // host is little endian
            bytes[b] = little ? tmp[b] : tmp[width - 1 - b];
        }
      return;
    }
  const bool is_signed = m_format.encoding() == Encoding::SIGNED;
  if (little && is_signed && width == 2)
    {
      float_to_s16le_clip16 (samples, bytes, n);
      return;
    }
  for (size_t i = 0; i < n; i++, bytes += width)
    {
      if (little && is_signed && width == 2)
        {
          /* native 16 bit path rounds at 16 bit (truncation toward zero) */
          const int16_t v = float_to_int_clip<16> (samples[i]);
          bytes[0] = v & 0xff;
          bytes[1] = (v >> 8) & 0xff;
          continue;
        }
      /* everything else: 32 bit value, most significant bytes are kept */
      uint32_t s = uint32_t (float_to_int_clip<32> (samples[i]));
      if (!is_signed)
        s ^= 0x80000000u;
      for (int b = 0; b < width; b++)
        {
          const int shift = 32 - 8 * width + 8 * b;      // little endian byte b
          bytes[little ? b : width - 1 - b] = (s >> shift) & 0xff;
        }
    }
}

void
RawConverter::from_raw (const unsigned char *bytes, float *samples, size_t n) const
{
  const int width = m_format.bit_depth() / 8;
  const bool little = m_format.endian() == RawFormat::LITTLE;
  if (m_format.encoding() == Encoding::FLOAT)
    {
      for (size_t i = 0; i < n; i++, bytes += width)
        {
          unsigned char tmp[8];
          for (int b = 0; b < width; b++)
            tmp[b] = little ? bytes[b] : bytes[width - 1 - b];
          if (width == 4)
            memcpy (samples + i, tmp, 4);
          else
            {
              double d;
              memcpy (&d, tmp, 8);
              samples[i] = d;
            }
        }
      return;
    }
  const bool is_signed = m_format.encoding() == Encoding::SIGNED;
  const float norm = 1.0 / 0x80000000LL;
  if (little && is_signed && width == 2)
    {
      s16le_to_float (bytes, samples, n);
      return;
    }
  for (size_t i = 0; i < n; i++, bytes += width)
    {
      uint32_t s = 0;                               // left-justified 32 bit value
      for (int b = 0; b < width; b++)
        s |= uint32_t (bytes[little ? b : width - 1 - b]) << (32 - 8 * width + 8 * b);
      if (!is_signed)
        s ^= 0x80000000u;
      samples[i] = int32_t (s) * norm;              // == int16 * (1 / 32768) for 16 bit input
    }
}

/* ---------------------------------------------------------------- raw streams */

static Error
open_in (const string& filename, FILE *& file, bool& close)
{
  if (filename == "-")
    {
      file = stdin;
      close = false;
    }
  else
    {
      file = fopen (filename.c_str(), "rb");
      if (!file)
        return Error (strerror (errno));
      close = true;
    }
  return Error::Code::NONE;
}

RawInputStream::~RawInputStream()
{
  if (m_close && m_file)
    fclose (m_file);
}

Error
RawInputStream::open (const string& filename, const RawFormat& format)
{
  if (!format.n_channels())
    return Error ("RawInputStream: input format: missing number of channels");
  if (!format.bit_depth())
    return Error ("RawInputStream: input format: missing bit depth");
  if (!format.sample_rate())
    return Error ("RawInputStream: input format: missing sample rate");
  Error err;
  m_conv.reset (RawConverter::create (format, err));
  if (err)
    return err;
  m_format = format;
  return open_in (filename, m_file, m_close);
}

static Error
read_converted (FILE *file, const RawConverter& conv, int width, int n_channels, vector<unsigned char>& bytes,
                vector<float>& samples, size_t count)
{
  const size_t frame_bytes = size_t (width) * n_channels;
  bytes.resize (count * frame_bytes);
  const size_t got = fread (bytes.data(), frame_bytes, count, file);
  if (ferror (file))
    return Error ("error reading sample data");
  samples.resize (got * n_channels);
  conv.from_raw (bytes.data(), samples.data(), samples.size());
  return Error::Code::NONE;
}

Error
RawInputStream::read_frames (vector<float>& samples, size_t count)
{
  return read_converted (m_file, *m_conv, m_format.bit_depth() / 8, m_format.n_channels(), m_bytes, samples, count);
}

RawOutputStream::~RawOutputStream()
{
  close();
}

Error
RawOutputStream::open (const string& filename, const RawFormat& format)
{
  if (!format.n_channels())
    return Error ("RawOutputStream: output format: missing number of channels");
  if (!format.bit_depth())
    return Error ("RawOutputStream: output format: missing bit depth");
  if (!format.sample_rate())
    return Error ("RawOutputStream: output format: missing sample rate");
  Error err;
  m_conv.reset (RawConverter::create (format, err));
  if (err)
    return err;
  if (filename == "-")
    {
      m_file = stdout;
      m_close = false;
    }
  else
    {
      m_file = fopen (filename.c_str(), "wb");
      if (!m_file)
        return Error (strerror (errno));
      m_close = true;
    }
  m_format = format;
  return Error::Code::NONE;
}

Error
RawOutputStream::write_frames (const vector<float>& samples)
{
  if (samples.empty())
    return Error::Code::NONE;
  vector<unsigned char> bytes (samples.size() * (m_format.bit_depth() / 8));
  m_conv->to_raw (samples.data(), bytes.data(), samples.size());
  if (fwrite (bytes.data(), 1, bytes.size(), m_file) != bytes.size())
    return Error ("write sample data failed");
  return Error::Code::NONE;
}

Error
RawOutputStream::close()
{
  if (m_file)
    {
      const bool bad = fflush (m_file) != 0;
      if (m_close)
        fclose (m_file);
      m_file = nullptr;
      if (bad)
        return Error ("error during flush");
    }
  return Error::Code::NONE;
}

/* ---------------------------------------------------------------- WAV input */

static uint32_t get_u32 (const unsigned char *b) { return b[0] | (b[1] << 8) | (b[2] << 16) | (uint32_t (b[3]) << 24); }
static uint16_t get_u16 (const unsigned char *b) { return b[0] | (b[1] << 8); }
static uint64_t get_u64 (const unsigned char *b) { return get_u32 (b) | (uint64_t (get_u32 (b + 4)) << 32); }

WavInputStream::~WavInputStream()
{
  if (m_close && m_file)
    fclose (m_file);
}

Error
WavInputStream::open (const string& filename, bool pipe_mode)
{
  m_pipe_mode = pipe_mode;
  Error err = open_in (filename, m_file, m_close);
  if (err)
    return err;
  auto bad = [&] (const string& msg) { return ferror (m_file) ? Error (string_printf ("wav input read error: %s", strerror (errno))) : Error (msg); };

  unsigned char riff[12];
  if (fread (riff, sizeof (riff), 1, m_file) != 1 || (memcmp (riff, "RIFF", 4) && memcmp (riff, "RF64", 4)) || memcmp (riff + 8, "WAVE", 4))
    return bad ("input file is not a valid wav file");
  const bool rf64 = !memcmp (riff, "RF64", 4);

  RawFormat format;
  bool have_fmt = false;
  uint64_t data_bytes = 0, ds64_data = 0;
  for (;;)
    {
      unsigned char chunk[8];
      if (fread (chunk, sizeof (chunk), 1, m_file) != 1)
        return bad ("wav input is incomplete (no data chunk found)");
      uint32_t size = get_u32 (chunk + 4);
      if (!memcmp (chunk, "fmt ", 4) && size >= 16 && size <= 64 * 1024 && !have_fmt)
        {
          vector<unsigned char> buf (size + (size & 1));
          if (fread (buf.data(), buf.size(), 1, m_file) != 1)
            return bad ("wav input is incomplete (error reading fmt chunk)");
          const int tag = get_u16 (&buf[0]);
          if (tag == 3)
            format.set_encoding (Encoding::FLOAT);
          else if (tag == 0xFFFE && size >= 40)
            {
              static const unsigned char pcm_guid[16] = { 1, 0, 0, 0, 0, 0, 0x10, 0, 0x80, 0, 0, 0xAA, 0, 0x38, 0x9B, 0x71 };
              static const unsigned char float_guid[16] = { 3, 0, 0, 0, 0, 0, 0x10, 0, 0x80, 0, 0, 0xAA, 0, 0x38, 0x9B, 0x71 };
              if (!memcmp (&buf[24], float_guid, 16) && !pipe_mode)
                format.set_encoding (Encoding::FLOAT);
              else if (memcmp (&buf[24], pcm_guid, 16))
                return Error ("wav input has unsupported extended format type, expected PCM");
            }
          else if (tag != 1)
            return Error (string_printf ("wav input has unsupported format type (%d), expected PCM", tag));
          format.set_channels (get_u16 (&buf[2]));
          format.set_sample_rate (get_u32 (&buf[4]));
          format.set_bit_depth (get_u16 (&buf[14]));
          if (format.bit_depth() == 8)
            format.set_encoding (Encoding::UNSIGNED);     // 8 bit wav is unsigned
          have_fmt = true;
        }
      else if (!memcmp (chunk, "ds64", 4) && size >= 24 && size <= 64 * 1024)
        {
          vector<unsigned char> buf (size + (size & 1));
          if (fread (buf.data(), buf.size(), 1, m_file) != 1)
            return bad ("wav input is incomplete (error reading ds64 chunk)");
          ds64_data = get_u64 (&buf[8]);
        }
      else if (!memcmp (chunk, "data", 4))
        {
          data_bytes = (size == 0xFFFFFFFFu && rf64) ? ds64_data : size;
          if (size == 0xFFFFFFFFu && !rf64)
            data_bytes = UINT64_MAX;                      // wav-pipe style header: length unknown
          break;
        }
      else
        {
          uint64_t todo = uint64_t (size) + (size & 1);
          char junk[4096];
          while (todo)
            {
              const size_t n = std::min<uint64_t> (todo, sizeof (junk));
              if (fread (junk, 1, n, m_file) != n)
                return bad ("wav input is incomplete (error skipping unknown chunk)");
              todo -= n;
            }
        }
    }
  if (!have_fmt)
    return Error ("wav input is incomplete (missing fmt chunk)");
  if (format.n_channels() <= 0 || format.sample_rate() <= 0)
    return Error ("wav input has an invalid fmt chunk");
  m_conv.reset (RawConverter::create (format, err));
  if (err)
    return err;
  m_format = format;
  const size_t frame_bytes = size_t (format.bit_depth() / 8) * format.n_channels();
  if (pipe_mode || data_bytes == UINT64_MAX)
    {
      m_n_frames = N_FRAMES_UNKNOWN;
      m_frames_left = N_FRAMES_UNKNOWN;
    }
  else
    {
      m_n_frames = data_bytes / frame_bytes;
      m_frames_left = m_n_frames;
    }
  return Error::Code::NONE;
}

Error
WavInputStream::read_frames (vector<float>& samples, size_t count)
{
  if (m_frames_left != N_FRAMES_UNKNOWN)
    count = std::min (count, m_frames_left);
  if (count == 0)
    {
      samples.clear();
      return Error::Code::NONE;
    }
  Error err = read_converted (m_file, *m_conv, m_format.bit_depth() / 8, m_format.n_channels(), m_bytes, samples, count);
  if (!err && m_frames_left != N_FRAMES_UNKNOWN)
    m_frames_left -= samples.size() / m_format.n_channels();
  return err;
}

Error
WavInputStream::read_raw_frames (unsigned char *bytes, size_t count, size_t *n_read, RawFormat *format)
{
  if (format)
    *format = m_format;
  *n_read = 0;
  if (m_frames_left != N_FRAMES_UNKNOWN)
    count = std::min (count, m_frames_left);
  if (count == 0)
    return Error::Code::NONE;
  const size_t frame_bytes = size_t (m_format.bit_depth() / 8) * m_format.n_channels();
  const size_t got = fread (bytes, frame_bytes, count, m_file);      /* whole frames only, as read_frames */
  if (ferror (m_file))
    return Error ("error reading sample data");
  if (m_frames_left != N_FRAMES_UNKNOWN)
    m_frames_left -= got;
  *n_read = got;
  return Error::Code::NONE;
}

/* ---------------------------------------------------------------- WAV output */

WavOutputStream::~WavOutputStream()
{
  close();
}

static void put_u16 (vector<unsigned char>& v, uint16_t u) { v.push_back (u); v.push_back (u >> 8); }
static void put_u32 (vector<unsigned char>& v, uint32_t u) { for (int i = 0; i < 4; i++) v.push_back (u >> (8 * i)); }
static void put_u64 (vector<unsigned char>& v, uint64_t u) { for (int i = 0; i < 8; i++) v.push_back (u >> (8 * i)); }
static void put_str (vector<unsigned char>& v, const char *s) { while (*s) v.push_back (*s++); }

void
WavOutputStream::write_header (uint64_t data_bytes, bool wav_pipe)
{
  vector<unsigned char> h;
  const uint64_t padded = data_bytes + (data_bytes & 1);
  if (m_rf64)
    {
      put_str (h, "RF64"); put_u32 (h, 0xFFFFFFFFu); put_str (h, "WAVE");
      put_str (h, "ds64"); put_u32 (h, 28);
      put_u64 (h, 72 + padded);                                     // riff size
      put_u64 (h, data_bytes);                                      // data size
      put_u64 (h, data_bytes / (uint64_t (m_bit_depth / 8) * m_n_channels));  // sample count
      put_u32 (h, 0);                                               // table length
    }
  else
    {
      put_str (h, "RIFF"); put_u32 (h, wav_pipe ? 0xFFFFFFFFu : uint32_t (36 + padded)); put_str (h, "WAVE");
    }
  put_str (h, "fmt "); put_u32 (h, 16);
  put_u16 (h, m_float ? 3 : 1);
  put_u16 (h, m_n_channels);
  put_u32 (h, m_sample_rate);
  put_u32 (h, m_sample_rate * m_n_channels * m_bit_depth / 8);
  put_u16 (h, m_n_channels * m_bit_depth / 8);
  put_u16 (h, m_bit_depth);
  put_str (h, "data"); put_u32 (h, (wav_pipe || m_rf64) ? 0xFFFFFFFFu : uint32_t (data_bytes));
  fwrite (h.data(), 1, h.size(), m_file);
}

static Error
check_depth (int bit_depth, Encoding encoding, const char *who)
{
  if (encoding == Encoding::FLOAT)
    {
      if (bit_depth != 32 && bit_depth != 64)
        return Error (string_printf ("%s: unsupported floating point bit depth %d", who, bit_depth));
    }
  else if (bit_depth != 16 && bit_depth != 24 && bit_depth != 32)
    return Error (string_printf ("%s: unsupported bit depth %d", who, bit_depth));
  return Error::Code::NONE;
}

Error
WavOutputStream::open_file (const string& filename, int n_channels, int sample_rate, int bit_depth, Encoding encoding, bool rf64)
{
  Error err = check_depth (bit_depth, encoding, "WavOutputStream::open");
  if (err)
    return err;
  m_file = fopen (filename.c_str(), "wb");
  if (!m_file)
    return Error (strerror (errno));
  m_close = true;
  m_rf64 = rf64;
  m_float = encoding == Encoding::FLOAT;
  m_bit_depth = bit_depth; m_sample_rate = sample_rate; m_n_channels = n_channels;
  write_header (0, false);
  m_open = true;
  return Error::Code::NONE;
}

Error
WavOutputStream::open_stdout (int n_channels, int sample_rate, int bit_depth, Encoding encoding, size_t n_frames, bool wav_pipe)
{
  Error err = check_depth (bit_depth, encoding, "StdoutWavOutputStream::open");
  if (err)
    return err;
  if (n_frames == AudioInputStream::N_FRAMES_UNKNOWN && !wav_pipe)
    return Error ("unable to write wav format to standard out without input length information");
  RawFormat format;
  format.set_bit_depth (bit_depth);
  format.set_encoding (encoding);
  m_conv.reset (RawConverter::create (format, err));
  if (err)
    return err;
  m_file = stdout;
  m_to_stdout = true;
  m_float = encoding == Encoding::FLOAT;
  m_bit_depth = bit_depth; m_sample_rate = sample_rate; m_n_channels = n_channels;
  m_data_bytes = uint64_t (n_frames) * n_channels * ((bit_depth + 7) / 8);     // announced size, decides the pad byte
  write_header (m_data_bytes, wav_pipe);
  if (ferror (stdout))
    return Error ("write wav header failed");
  m_open = true;
  return Error::Code::NONE;
}

Error
WavOutputStream::write_frames (const vector<float>& samples)
{
  if (samples.empty())
    return Error::Code::NONE;
  const int width = m_bit_depth / 8;
  vector<unsigned char> bytes (samples.size() * width);
  if (m_to_stdout)
    m_conv->to_raw (samples.data(), bytes.data(), samples.size());
  else if (!m_float && m_bit_depth == 16)
    {
      float_to_s16le_msb (samples.data(), bytes.data(), samples.size());
      m_data_bytes += bytes.size();
    }
  else
    {
      unsigned char *p = bytes.data();
      for (float s : samples)
        {
          if (m_float)
            {
              if (width == 4) { const float f = float_clip (s); memcpy (p, &f, 4); }
              else            { const double d = float_clip (s); memcpy (p, &d, 8); }
            }
          else
            {
              /* libsndfile int API: 32 bit value, the file keeps the most significant bits */
              const uint32_t v = uint32_t (float_to_int_clip<32> (s) >> (32 - m_bit_depth));
              for (int b = 0; b < width; b++)
                p[b] = (v >> (8 * b)) & 0xff;
            }
          p += width;
        }
      m_data_bytes += bytes.size();
    }
  if (fwrite (bytes.data(), 1, bytes.size(), m_file) != bytes.size())
    return Error (string_printf ("write sample data failed (%s)", strerror (errno)));
  return Error::Code::NONE;
}

Error
WavOutputStream::close()
{
  if (!m_open)
    return Error::Code::NONE;
  m_open = false;
  if (m_data_bytes & 1)
    fputc (0, m_file);
  if (!m_to_stdout)
    {
      fseek (m_file, 0, SEEK_SET);
      write_header (m_data_bytes, false);
    }
  bool bad = fflush (m_file) != 0 || ferror (m_file);
  if (m_close)
    bad |= fclose (m_file) != 0;
  m_file = nullptr;
  return bad ? Error ("error during flush") : Error (Error::Code::NONE);
}

/* ---------------------------------------------------------------- factories (src/audiostream.cc:34-121) */

std::unique_ptr<AudioInputStream>
AudioInputStream::create (const string& filename, Error& err)
{
  std::unique_ptr<AudioInputStream> in_stream;
  if (Params::input_format == Format::AUTO || Params::input_format == Format::WAV_PIPE)
    {
      WavInputStream *w = new WavInputStream();
      in_stream.reset (w);
      err = w->open (filename, Params::input_format == Format::WAV_PIPE);
    }
  else if (Params::input_format == Format::RAW)
    {
      RawInputStream *r = new RawInputStream();
      in_stream.reset (r);
      err = r->open (filename, Params::raw_input_format);
    }
  else
    err = Error ("selected format is not supported as input format");
  if (err)
    return nullptr;
  return in_stream;
}

std::unique_ptr<AudioOutputStream>
AudioOutputStream::create (const string& filename, int n_channels, int sample_rate, int bit_depth, Encoding encoding, size_t n_frames, Error& err)
{
  std::unique_ptr<AudioOutputStream> out_stream;
  if (Params::output_format == Format::RAW)
    {
      RawOutputStream *r = new RawOutputStream();
      out_stream.reset (r);
      err = r->open (filename, Params::raw_output_format);
    }
  else
    {
      WavOutputStream *w = new WavOutputStream();
      out_stream.reset (w);
      if (filename == "-")
        err = w->open_stdout (n_channels, sample_rate, bit_depth, encoding, n_frames, Params::output_format == Format::WAV_PIPE);
      else
        err = w->open_file (filename, n_channels, sample_rate, bit_depth, encoding, Params::output_format == Format::RF64);
    }
  if (err)
    return nullptr;
  return out_stream;
}

/* ---------------------------------------------------------------- WavData */

Error
WavData::load (const string& filename)
{
  Error err;
  std::unique_ptr<AudioInputStream> in_stream = AudioInputStream::create (filename, err);
  if (err)
    return err;
  return load (in_stream.get());
}

Error
WavData::load (AudioInputStream *in_stream)
{
  m_samples.clear();
  if (in_stream->n_frames() != AudioInputStream::N_FRAMES_UNKNOWN)
    m_samples.reserve (in_stream->n_frames() * in_stream->n_channels());
  vector<float> buffer;
  for (;;)
    {
      Error err = in_stream->read_frames (buffer, 65536);
      if (err)
        return err;
      if (buffer.empty())
        break;
      m_samples.insert (m_samples.end(), buffer.begin(), buffer.end());
    }
  m_sample_rate = in_stream->sample_rate();
  m_n_channels  = in_stream->n_channels();
  m_bit_depth   = in_stream->bit_depth();
  return Error::Code::NONE;
}

Error
WavData::save (const string& filename) const
{
  Error err;
  std::unique_ptr<AudioOutputStream> out = AudioOutputStream::create (filename, m_n_channels, m_sample_rate, m_bit_depth, Encoding::SIGNED, n_frames(), err);
  if (err)
    return err;
  err = out->write_frames (m_samples);
  if (err)
    return err;
  return out->close();
}
