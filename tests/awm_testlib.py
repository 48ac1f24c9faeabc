"""Shared helpers for the parity tests: oracle tables -> C-ABI structs, synthetic signals."""
from __future__ import annotations

import numpy as np

import awm_oracle as O
from audiowmark_b200 import capi

PAYLOAD = "0123456789abcdef0011223344556677"


def sync_entries(key, mode, P):
    sb = O.get_sync_bits(key, mode, P)
    ent = np.zeros(len(sb.frame), capi.SYNC_ENTRY)
    ent["frame"] = sb.frame
    ent["up"] = sb.up.reshape(-1, P.bands_per_frame)
    ent["down"] = sb.down.reshape(-1, P.bands_per_frame)
    return ent, sb.off.astype(np.int32)


def mix_entries(key, P):
    m = O.gen_mix_entries(key, P)
    ent = np.zeros(len(m), capi.MIX_ENTRY)
    ent["frame"] = [e[0] for e in m]
    ent["up"] = [e[1] for e in m]
    ent["down"] = [e[2] for e in m]
    n_coded = O.conv_code_size(O.A, P.payload_size)
    order = np.array(O.randomize_bit_order(key, list(range(n_coded)), True), np.uint16)
    return ent, order


def frame_mod_ab(key, payload, P):
    bitvec = O.parse_payload(payload, P)
    return np.stack([O.init_frame_mod(key, 0, bitvec, P), O.init_frame_mod(key, 1, bitvec, P)])


def setup_ctx(ctx, key, P, payload=None, key_slot=0):
    """Feed one key's tables (built by the ORACLE, so kernels are tested independently of host/ table code)."""
    for mode in (capi.MODE_BLOCK, capi.MODE_CLIP):
        ent, off = sync_entries(key, mode, P)
        ctx.set_sync_tables(key_slot, mode, ent, off)
    ent, order = mix_entries(key, P)
    ctx.set_mix_tables(key_slot, ent, order, P.frames_per_bit, O.frames_per_block(P))
    if payload is not None:
        ctx.set_embed_tables(frame_mod_ab(key, payload, P))


def noise(seconds, channels=2, seed=1234, amp=0.5):
    rng = np.random.default_rng(seed)
    n = int(seconds * 44100)
    return ((rng.random((n, channels), dtype=np.float32) - 0.5) * (2 * amp)).astype(np.float32)


# --------------------------------------------------------------------------- deterministic "music-like" signals
# Seeded numpy in float64, returned on the 16 bit grid (float32, as a 16 bit file reads back); where results for them are stored,
# so is the SHA-256 of the int16 samples, so a box whose numpy / scipy computes a different signal fails loudly.
# Tones are periodic in samples: their phase is looked up from the integer sample index, never computed as sin of a large argument.

RATE = 44100

# (cycles, period): a tone with `cycles` periods every `period` samples; bin k of the 1024 point analysis is k * 44100 / 1024 Hz,
# the sync / data bands are bins 20..100
MUSIC_TONES = ((40, 1024), (71, 1024),        # on the bin centres k = 40, 71
               (105, 2048), (177, 2048),      # half-way between bins: k = 52.5, 88.5
               (11, 2205),                    # 220 Hz, below the band
               (20, 147))                     # 6 kHz, above it
TONE_475 = (95, 2048)                         # k = 47.5: half-way between two in-band bins


def db(v):
    return 10.0 ** (v / 20.0)


def periodic_tone(n, cycles, period, phase_num=0, channels=1):
    """sin(2 pi (t * cycles / period + phase)) for t = 0..n-1, phase = (phase_num + channel) / 7 of a cycle -> float64 [n, channels]"""
    t = np.arange(n, dtype=np.int64)
    table = np.sin(2 * np.pi * np.arange(period, dtype=np.float64) / period)
    out = np.empty((n, channels))
    for c in range(channels):
        off = (period * (phase_num + c)) // 7
        out[:, c] = table[(t * cycles + off) % period]
    return out


def pink(n, channels, rng):
    """independent 1/f noise per channel: seeded white noise through a fixed 3-pole / 3-zero IIR with a roughly
    -3 dB/octave response, normalised to RMS 1"""
    from scipy.signal import lfilter
    b = [0.049922035, -0.095993537, 0.050612699, -0.004408786]
    a = [1.0, -2.494956002, 2.017265875, -0.522189400]
    w = rng.standard_normal((n + 4096, channels))
    p = lfilter(b, a, w, axis=0)[4096:]              # the filter's start-up transient is cut off
    return p / np.sqrt(np.mean(p * p, axis=0))


def to16(x):
    """float64 -> the 16 bit grid (clipped like a 16 bit file write) -> float32"""
    return O.int16_to_float(O.quantize_sndfile16(np.asarray(x, np.float64).astype(np.float32)))


def music_f64(seconds, channels=2, seed=1):
    """pink noise at -20 dBFS RMS per channel plus six steady -12 dBFS tones shared by all channels (per-channel phases);
    the sum is scaled to a -1 dBFS peak, so the tones end up near -16 dBFS"""
    n = int(seconds * RATE)
    rng = np.random.default_rng(seed)
    x = db(-20) * pink(n, channels, rng)
    for j, (cycles, period) in enumerate(MUSIC_TONES):
        x += db(-12) * periodic_tone(n, cycles, period, phase_num=j, channels=channels)
    return x * (db(-1) / np.abs(x).max())


def music(seconds, channels=2, seed=1):
    return to16(music_f64(seconds, channels, seed))


def tone(seconds, channels=2, seed=2):
    """one -6 dBFS tone half-way between two in-band bins over a noise floor of 1 LSB RMS: the widest in-band dynamic range a
    16 bit file holds, and the input on which the sliding DFT's cancellation errors are largest"""
    n = int(seconds * RATE)
    rng = np.random.default_rng(seed)
    x = db(-6) * periodic_tone(n, *TONE_475, channels=channels) + rng.standard_normal((n, channels)) / 32768
    return to16(x)


def quiet(seconds, channels=2, seed=3):
    """music at a -60 dBFS peak: a few dozen LSB"""
    x = music_f64(seconds, channels, seed)
    return to16(x * (db(-60) / np.abs(x).max()))


def dc_clip(seconds, channels=2, seed=4):
    """music + 0.3 DC, amplified until 1 % of the samples exceed full scale, hard clipped"""
    x = music_f64(seconds, channels, seed)
    lo, hi = 0.5, 8.0                                  # bisect the gain: fraction of |g x + 0.3| > 1 is monotonic in g
    for _ in range(60):
        g = 0.5 * (lo + hi)
        if np.mean(np.abs(g * x + 0.3) > 1.0) < 0.01:
            lo = g
        else:
            hi = g
    return to16(np.clip(lo * x + 0.3, -1.0, 1.0))


def one_sided(seconds, kind, seed=5):
    """stereo from one music channel L: kind "zero" (R = 0), "m50" (R = L at -50 dB: tens of LSB), "same" (R = L), "neg" (R = -L)"""
    L = music_f64(seconds, 1, seed)[:, 0]
    R = {"zero": 0.0 * L, "m50": db(-50) * L, "same": L, "neg": -L}[kind]
    return to16(np.stack([L, R], axis=1))


SIGNALS = {"music": music, "tone": tone, "quiet": quiet, "dc_clip": dc_clip, "one_sided": one_sided}


def signal(spec):
    """spec = {"fn": name in SIGNALS, "args": keyword arguments} (how tests/golden/golden_large.json names its inputs)"""
    return SIGNALS[spec["fn"]](**spec["args"])


def rms(x):
    x = np.asarray(x, np.float64)
    return float(np.sqrt(np.mean(x * x))) if x.size else 0.0


_SPEED_CACHE = {}


def watermarked_noise(seconds, payload="f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0"):
    """reference test signal: keyed noise (test-gen-noise), watermarked by the oracle, on the 16 bit grid"""
    k = ("wm", seconds, payload)
    if k not in _SPEED_CACHE:
        x = O.int16_to_float(O.quantize_sndfile16(O.gen_noise(seconds)))
        _SPEED_CACHE[k] = O.int16_to_float(O.quantize_sndfile16(O.embed(x, O.Key(), payload, O.Params()).samples))
    return _SPEED_CACHE[k]


def cli_float(v):
    """the reference CLI parses every floating point argument with strtof (src/audiowmark.cc:188-199)"""
    return float(np.float32(v))


def speed_changed(seconds, speed):
    """tests/detect-speed-test.sh input: test-change-speed = resample_ratio (1 / speed), saved as 16 bit"""
    k = ("sp", seconds, speed)
    if k not in _SPEED_CACHE:
        y = watermarked_noise(seconds)
        _SPEED_CACHE[k] = O.int16_to_float(O.quantize_sndfile16(O.resample_ratio(y, 1 / cli_float(speed))))
    return _SPEED_CACHE[k]
