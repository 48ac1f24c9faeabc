"""Streamed `get` / `cmp`: WAV samples read chunk by chunk into two host buffers and decoded on the device (k_wav_to_f32).

- the device decode (awm_pcm_bind_wav, awm_pcm_prefetch_wav) equals the host's RawConverter bit for bit for every WAV sample format
- `get` / `cmp` print what the reference prints for the same marked signal stored as 8/16/24/32 bit PCM, float32, float64, RF64 and
  WAVE_FORMAT_EXTENSIBLE (tests/golden/stream_ref.json, made by tests/golden/make_golden_stream.py), from a file and from stdin
- the streamed CLI equals the whole-buffer path (hostapi.get on host-decoded floats, pinned to the reference) byte for byte
- host memory does not grow with the input length"""
import hashlib
import json
import os
import struct
import subprocess
import tempfile

import numpy as np
import pytest

import awm_oracle as O
import awm_testlib as T

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden", "stream_ref.json")
PAYLOAD = "f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0"
RATE = 44100
FORMATS = [(8, False), (16, False), (24, False), (32, False), (32, True), (64, True)]      # (bits, is_float)

# ---------------------------------------------------------------- WAV files (shared with tests/golden/make_golden_stream.py)


def encode(x, bits, is_float, dither_seed=None):
    """float32 [n, ch] -> stored sample bytes as the reference's writer stores them: integers = float_to_int_clip<32> with the top
    `bits` kept (8 bit: + 128, unsigned); float32 as is; float64 = x plus a seeded 2^-30 dither, so that reading has to round"""
    x = np.asarray(x, np.float32)
    if is_float and bits == 32:
        return x.astype("<f4").tobytes()
    if is_float:
        d = x.astype(np.float64)
        if dither_seed is not None:
            d = d + np.random.default_rng(dither_seed).uniform(-2.0 ** -30, 2.0 ** -30, d.shape)
        return d.astype("<f8").tobytes()
    v = O.float_to_int_clip(x, 32).astype(np.int64) >> (32 - bits)
    if bits == 8:
        return (v + 128).astype(np.uint8).tobytes()
    if bits == 24:
        u = (v & 0xFFFFFF).astype("<u4").view(np.uint8).reshape(-1, 4)[:, :3]
        return np.ascontiguousarray(u).tobytes()
    return v.astype({16: "<i2", 32: "<i4"}[bits]).tobytes()


def wav_file(data: bytes, channels, bits, is_float, rate=RATE, container="riff"):
    """RIFF (fmt tag 1 / 3), "rf64" (RF64 + ds64) or "extensible" (WAVE_FORMAT_EXTENSIBLE) around the sample bytes"""
    block = channels * bits // 8
    tag = 3 if is_float else 1
    fmt = struct.pack("<HHIIHH", tag, channels, rate, rate * block, block, bits)
    if container == "extensible":
        guid = bytes([tag, 0, 0, 0, 0, 0, 0x10, 0, 0x80, 0, 0, 0xAA, 0, 0x38, 0x9B, 0x71])
        fmt = struct.pack("<HHIIHH", 0xFFFE, channels, rate, rate * block, block, bits) + struct.pack("<HHI", 22, bits, 0) + guid
    pad = b"\0" if len(data) & 1 else b""
    body = b"fmt " + struct.pack("<I", len(fmt)) + fmt
    if container == "rf64":
        ds64 = struct.pack("<QQQI", 4 + 36 + 8 + len(body) + 8 + len(data) + len(pad), len(data), len(data) // block, 0)
        return b"RF64" + struct.pack("<I", 0xFFFFFFFF) + b"WAVE" + b"ds64" + struct.pack("<I", len(ds64)) + ds64 + body + \
            b"data" + struct.pack("<I", 0xFFFFFFFF) + data + pad
    return b"RIFF" + struct.pack("<I", 4 + len(body) + 8 + len(data) + len(pad)) + b"WAVE" + body + b"data" + struct.pack("<I", len(data)) + data + pad


# name -> (bits, is_float, container)
STREAM_CASES = {
    "u8": (8, False, "riff"), "s16": (16, False, "riff"), "s24": (24, False, "riff"), "s32": (32, False, "riff"),
    "f32": (32, True, "riff"), "f64": (64, True, "riff"), "rf64_s24": (24, False, "rf64"), "ext_s24": (24, False, "extensible"),
}
STREAM_SIGNAL = {"fn": "music", "args": {"seconds": 130, "channels": 2, "seed": 11}}


def marked_signal():
    """the seeded 130 s music signal marked by the oracle's add (CPU)"""
    x = T.signal(STREAM_SIGNAL)
    return O.embed(x, O.Key(), PAYLOAD, O.Params()).samples.astype(np.float32)


def stream_files(y):
    """name -> bytes of the WAV file"""
    out = {}
    for name, (bits, is_float, container) in STREAM_CASES.items():
        out[name] = wav_file(encode(y, bits, is_float, dither_seed=7), y.shape[1], bits, is_float, container=container)
    return out


def sha(b: bytes) -> str:
    return hashlib.sha256(b).hexdigest()


def cli():
    from audiowmark_b200 import hostapi as H
    return H.CLI_PATH


# ---------------------------------------------------------------- 1. the device decode is exact


def special_bytes(bits, is_float, rng, n):
    """n random samples with the extremes of the format mixed in"""
    if not is_float:
        extremes = {8: [0, 255, 128, 127, 1], 16: [-32768, 32767, 0, -1, 1], 24: [-0x800000, 0x7FFFFF, 0, -1, 1],
                    32: [-2 ** 31, 2 ** 31 - 1, 0, -1, 1, 0x7FFFFFC0, 0x40000041]}[bits]
        raw = rng.integers(0, 256, n * bits // 8, dtype=np.uint8)
        ext = np.array(extremes, np.int64) & ((1 << bits) - 1)
        for j, e in enumerate(ext):
            pos = (j * 7 + 3) % n
            raw[pos * bits // 8:(pos + 1) * bits // 8] = np.frombuffer(int(e).to_bytes(bits // 8, "little"), np.uint8)
        return raw
    if bits == 32:
        special = np.array([0x7F800000, 0xFF800000, 0x7FC00000, 0x7FC12345, 0x7F800001, 0xFFC00001, 0x00000001, 0x807FFFFF,
                            0x3FC00000, 0x80000000], np.uint32)                 # +-Inf, NaNs, denormals, 1.5, -0
        v = rng.integers(0, 2 ** 32, n, dtype=np.uint64).astype(np.uint32)
    else:
        special = np.array([0x7FF0000000000000, 0xFFF0000000000000, 0x7FF8000000000000, 0x7FF8000000000001, 0x7FF0000000000001,
                            0xFFFC0000DEADBEEF, 0x0000000000000001, 0x3810000000000000, 0x3800000000000001, 0x3FF8000000000000,
                            0x3FF0000010000000, 0x3FF0000030000000, 0x7FE0000000000000, 0x47EFFFFFF0000000], np.uint64)
        v = rng.integers(0, 2 ** 63, n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, n, dtype=np.uint64)
        # random doubles are mostly far outside the float range: half of them get a float-sized exponent
        e = rng.integers(0x380, 0x47F, n, dtype=np.uint64)
        keep = rng.integers(0, 2, n).astype(bool)
        v[keep] = (v[keep] & np.uint64(0x800FFFFFFFFFFFFF)) | (e[keep] << np.uint64(52))
    v[np.arange(len(special)) * 5 % n] = special
    return v.view(np.uint8)


@pytest.fixture(scope="module")
def ctx():
    from audiowmark_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def bound_floats(ctx):
    p, n, ch = ctx.pcm_device()
    assert p
    return ctx.copy_to_host(np.empty(n * ch, np.float32), p)


@pytest.mark.parametrize("bits,is_float", FORMATS)
@pytest.mark.parametrize("channels", [1, 2, 3])
def test_wav_decode_exact(ctx, bits, is_float, channels):
    import torch
    from audiowmark_b200 import hostapi as H
    rng = np.random.default_rng(bits * 10 + channels)
    n_frames = 1001                                    # odd: not a multiple of the four samples a thread decodes
    raw = special_bytes(bits, is_float, rng, n_frames * channels)
    want = H.wav_decode_host(raw, bits, is_float).view(np.uint32)
    # host buffer at odd addresses (copied to an aligned device buffer)
    for off in (0, 1, 3):
        buf = np.zeros(raw.nbytes + 8, np.uint8)
        buf[off:off + raw.nbytes] = raw
        ctx.pcm_bind_wav(buf, bits, is_float, n_frames, channels, offset=off)
        got = bound_floats(ctx).view(np.uint32)
        assert np.array_equal(got, want), (off, np.flatnonzero(got != want)[:5])
    # device buffer at every alignment: the kernel reads the words around the samples
    dev = torch.from_numpy(np.concatenate([np.zeros(16, np.uint8), raw, np.zeros(16, np.uint8)])).cuda()
    for off in range(16):
        d = torch.zeros(raw.nbytes + 32, dtype=torch.uint8, device="cuda")
        d[off:off + raw.nbytes] = dev[16:16 + raw.nbytes]
        torch.cuda.synchronize()
        for n in (n_frames, 1, 2, 5):                   # short spans: the byte-by-byte tail alone
            ctx.pcm_bind_wav(d.data_ptr(), bits, is_float, n, channels, offset=off)
            got = bound_floats(ctx).view(np.uint32)
            assert np.array_equal(got, want[:n * channels]), (off, n, np.flatnonzero(got != want[:n * channels])[:5])
    # zero padding in front: the floats land at an odd position of the device buffer
    ctx.pcm_bind_wav(raw, bits, is_float, n_frames, channels, pad_start=1, pad_end=2)
    got = bound_floats(ctx).view(np.uint32)
    assert np.array_equal(got[channels:channels + want.size], want) and not got[:channels].any() and not got[channels + want.size:].any()


@pytest.mark.parametrize("bits,is_float", [(16, False), (24, False), (64, True)])
@pytest.mark.parametrize("bind_between", [True, False])
def test_wav_prefetch_overlap(ctx, bits, is_float, bind_between):
    """a span whose head is the tail of the span before, in another host buffer: same floats as a plain bind of the whole span"""
    rng = np.random.default_rng(bits)
    ch, n_a, n_b, head = 2, 5003, 4001, 1234
    fb = ch * bits // 8
    whole = special_bytes(bits, is_float, rng, (n_a + n_b - head) * ch)
    a = np.ascontiguousarray(whole[:n_a * fb])
    b_new = np.ascontiguousarray(whole[n_a * fb:])                  # only the frames after the head
    b_full = np.ascontiguousarray(whole[(n_a - head) * fb:])
    ctx.pcm_bind_wav(b_full, bits, is_float, n_b, ch)
    want = bound_floats(ctx).view(np.uint32)
    ctx.pcm_prefetch_wav(a, bits, is_float, n_a, ch)
    if bind_between:
        ctx.pcm_bind_wav(a, bits, is_float, n_a, ch)
    ctx.pcm_prefetch_wav(b_new, bits, is_float, n_b, ch, head_frames=head)
    if not bind_between:
        ctx.pcm_bind_wav(a, bits, is_float, n_a, ch)
        assert np.array_equal(bound_floats(ctx).view(np.uint32), H_decode(a, bits, is_float))
    ctx.pcm_bind_wav(b_new, bits, is_float, n_b, ch)
    assert np.array_equal(bound_floats(ctx).view(np.uint32), want)


def H_decode(raw, bits, is_float):
    from audiowmark_b200 import hostapi as H
    return H.wav_decode_host(raw, bits, is_float).view(np.uint32)


# ---------------------------------------------------------------- 2. parity with the reference for each WAV format


@pytest.fixture(scope="module")
def stream_golden():
    G = json.load(open(GOLDEN))
    assert G["signal"] == STREAM_SIGNAL and G["payload"] == PAYLOAD
    files = stream_files(marked_signal())
    for name, data in files.items():
        assert sha(data) == G["cases"][name]["sha256"], name
    return G, files


@pytest.mark.parametrize("name", sorted(STREAM_CASES))
@pytest.mark.parametrize("cmd", ["get", "cmp"])
def test_stream_formats_vs_reference(stream_golden, name, cmd):
    G, files = stream_golden
    want = G["cases"][name][cmd]
    args = [PAYLOAD] if cmd == "cmp" else []
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, name + ".wav")
        open(path, "wb").write(files[name])
        p = subprocess.run([cli(), cmd, path] + args, capture_output=True)
        assert (p.returncode, p.stdout.decode()) == (want["returncode"], want["stdout"]), p.stderr.decode()
    p = subprocess.run([cli(), cmd, "-"] + args, input=files[name], capture_output=True)
    assert (p.returncode, p.stdout.decode()) == (want["returncode"], want["stdout"]), p.stderr.decode()


# ---------------------------------------------------------------- 3. streamed == whole buffer


@pytest.fixture(scope="module")
def marked25():
    from audiowmark_b200 import hostapi as H
    H.set_params()
    x = T.noise(25 * 60.0, 2, seed=2501, amp=0.3)
    return H.add(x, PAYLOAD)


def whole_buffer(y, bits, extra_speed=False, seconds=None):
    """hostapi.get on the floats the host decodes from the stored bytes, chunk size 10 min"""
    from audiowmark_b200 import hostapi as H
    data = encode(y, bits, False)
    x = H.wav_decode_host(data, bits).reshape(-1, y.shape[1])
    if seconds is not None:
        x = x[:seconds * RATE]
    H.set_params(chunk_size_min=10)
    H.set_speed_params(detect_speed=extra_speed)
    try:
        return data, H.get(x, parse=False)
    finally:
        H.set_speed_params()
        H.set_params()


def cli_get_json(data, channels, bits, *opts):
    wav = wav_file(data, channels, bits, False)
    p = subprocess.run([cli(), "get", "--chunk-size", "10", *opts, "--json", "-", "-"], input=wav, capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    return p.stdout.decode()


@pytest.mark.parametrize("bits", [16, 24])
@pytest.mark.parametrize("frames", [25 * 60 * RATE, 10 * 60 * RATE, 10 * 60 * RATE + 1], ids=["25min", "10min", "10min+1"])
def test_streamed_equals_whole_buffer(marked25, bits, frames):
    from audiowmark_b200 import hostapi as H
    y = marked25[:frames]
    data, want = whole_buffer(y, bits)
    assert json.loads(want)["matches"]
    assert cli_get_json(data, 2, bits) == want
    H.set_params(chunk_size_min=10)
    try:                                              # the same loader over a memory buffer, read in pipe-sized pieces
        assert H.get_wav_bytes(data, 2, bits, chunk_buffer=12345, parse=False) == want
    finally:
        H.set_params()


@pytest.mark.parametrize("bits", [16, 24])
def test_streamed_detect_speed_clip(marked25, bits):
    y = marked25[100 * RATE:130 * RATE]
    data, want = whole_buffer(y, bits, extra_speed=True)
    assert cli_get_json(data, 2, bits, "--detect-speed") == want


@pytest.mark.parametrize("bits", [16, 24])
def test_streamed_test_truncate(marked25, bits):
    data, want = whole_buffer(marked25, bits, seconds=300)
    assert cli_get_json(data, 2, bits, "--test-truncate", "300") == want


# ---------------------------------------------------------------- 4. host memory is bounded


def peak_rss_mb(args):
    """run args to the end; its peak resident set size from wait4's rusage"""
    with tempfile.TemporaryFile() as err:
        p = subprocess.Popen(args, stdout=subprocess.DEVNULL, stderr=err)
        _, status, ru = os.wait4(p.pid, 0)
        p.returncode = os.waitstatus_to_exitcode(status)
        err.seek(0)
        assert p.returncode == 0, err.read().decode()
    return ru.ru_maxrss / 1024.0


def test_streamed_memory_bounded():
    rng = np.random.default_rng(40)
    peaks = {}
    with tempfile.TemporaryDirectory() as tmp:
        for minutes in (40, 12):
            path = os.path.join(tmp, "m%d.wav" % minutes)
            pcm = rng.integers(-3000, 3000, (minutes * 60 * RATE, 2), dtype=np.int16)
            open(path, "wb").write(wav_file(pcm.astype("<i2").tobytes(), 2, 16, False))
            del pcm
            peaks[minutes] = peak_rss_mb([cli(), "get", "--chunk-size", "10", path])
            os.unlink(path)
    print("peak RSS MB:", peaks)
    assert abs(peaks[40] - peaks[12]) < 64, peaks
