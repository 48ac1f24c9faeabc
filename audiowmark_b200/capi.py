"""ctypes binding of the C ABI (include/awm_b200.h) exported by lib/libawm_b200.so.

Thin by design: arguments are numpy arrays (host) or raw device pointers (ints, e.g.
torch.Tensor.data_ptr()).  Nothing here computes; if the CUDA library is missing or no
device is usable every call fails loudly -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libawm_b200.so")

FRAME = 1024
N_BANDS = 81
MODE_BLOCK, MODE_CLIP = 0, 1
BLOCK_A, BLOCK_B, BLOCK_AB = 0, 1, 2

SYNC_ENTRY = np.dtype([("frame", "<u2"), ("up", "u1", (30,)), ("down", "u1", (30,))])       # awm_sync_entry
MIX_ENTRY = np.dtype([("frame", "<u2"), ("up", "u1"), ("down", "u1")])                      # awm_mix_entry
SEARCH_SCORE = np.dtype([("index", "<u8"), ("raw_quality", "<f8"), ("local_mean", "<f8")])  # awm_search_score

EXPORTS = [
    "awm_create", "awm_destroy", "awm_last_error", "awm_launch_count", "awm_stream", "awm_synchronize",
    "awm_profile_enable", "awm_profile_report", "awm_host_alloc", "awm_host_free",
    "awm_fft_r2c", "awm_fft_c2r", "awm_set_embed_tables", "awm_set_sync_tables", "awm_set_mix_tables",
    "awm_pcm_bind", "awm_pcm_prefetch", "awm_embed", "awm_sync_approx", "awm_sync_peaks", "awm_sync_refine", "awm_sync_refine_offsets", "awm_decode_blocks", "awm_viterbi",
    "awm_resample", "awm_pcm_push_resampled", "awm_pcm_pop", "awm_copy_to_host", "awm_is_device_pointer", "awm_speed_scan", "awm_embed_resampled", "awm_gather", "awm_pcm_bind_s16", "awm_pcm_prefetch_s16", "awm_pcm_device", "awm_embed_s16", "awm_embed_window", "awm_pcm_stage", "awm_pcm_stage_wait", "awm_dist_unique_id", "awm_dist_init", "awm_dist_world", "awm_dist_allgather",
    "awm_pcm_bind_wav", "awm_pcm_prefetch_wav",
]

_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(the CUDA extension is mandatory, there is no CPU fallback)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        lib.awm_last_error.restype = ctypes.c_char_p
        lib.awm_launch_count.restype = ctypes.c_uint64
        lib.awm_stream.restype = ctypes.c_void_p
        _lib = lib
    return _lib


def _ptr(x):
    """numpy array -> host pointer, int -> device pointer."""
    if x is None:
        return ctypes.c_void_p(0)
    if isinstance(x, (int, np.integer)):
        return ctypes.c_void_p(int(x))
    assert x.flags["C_CONTIGUOUS"]
    return x.ctypes.data_as(ctypes.c_void_p)


class AwmError(RuntimeError):
    pass


class WavFormat(ctypes.Structure):
    """awm_wav_format: how WAV samples are stored (8 bit unsigned, 16/24/32 bit signed, 32/64 bit float; little endian)"""
    _fields_ = [("bits", ctypes.c_int), ("is_float", ctypes.c_int)]


class Context:
    """One awm_ctx (device + stream)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        h = ctypes.c_void_p()
        rc = self.lib.awm_create(ctypes.c_int(device), ctypes.byref(h))
        if rc != 0 or not h:
            raise AwmError("awm_create failed (rc=%d): no usable CUDA device; this package has no CPU fallback" % rc)
        self.h = h

    @classmethod
    def from_handle(cls, handle):
        """non-owning view of an existing awm_ctx* (the host library's engine context)"""
        self = cls.__new__(cls)
        self.lib = load()
        self.h = ctypes.c_void_p(handle)
        self._borrowed = True
        if not handle:
            raise AwmError("no GPU context (a CUDA device is required, there is no CPU fallback)")
        return self

    def close(self):
        if getattr(self, "h", None) and not getattr(self, "_borrowed", False):
            self.lib.awm_destroy(self.h)
        self.h = None

    __del__ = close

    def _ck(self, rc):
        if rc != 0:
            raise AwmError(self.lib.awm_last_error(self.h).decode())

    @property
    def launches(self) -> int:
        return int(self.lib.awm_launch_count(self.h))

    @property
    def stream(self) -> int:
        return int(self.lib.awm_stream(self.h) or 0)

    def synchronize(self):
        self._ck(self.lib.awm_synchronize(self.h))

    def profile_enable(self, on=True):
        self._ck(self.lib.awm_profile_enable(self.h, ctypes.c_int(1 if on else 0)))

    def profile_report(self) -> dict:
        import json
        buf = ctypes.create_string_buffer(1 << 16)
        self._ck(self.lib.awm_profile_report(self.h, buf, ctypes.c_size_t(len(buf))))
        return json.loads(buf.value.decode())

    # ---- FFTProcessor
    def fft_r2c(self, x: np.ndarray) -> np.ndarray:
        x = np.ascontiguousarray(x, np.float32).reshape(-1, FRAME)
        out = np.empty((x.shape[0], FRAME + 2), np.float32)
        self._ck(self.lib.awm_fft_r2c(self.h, _ptr(x), _ptr(out), ctypes.c_size_t(x.shape[0]), ctypes.c_int(FRAME)))
        return out.view(np.complex64)

    def fft_c2r(self, spec: np.ndarray) -> np.ndarray:
        s = np.ascontiguousarray(spec, np.complex64).reshape(-1, FRAME // 2 + 1).view(np.float32)
        out = np.empty((s.shape[0], FRAME), np.float32)
        self._ck(self.lib.awm_fft_c2r(self.h, _ptr(s), _ptr(out), ctypes.c_size_t(s.shape[0]), ctypes.c_int(FRAME)))
        return out

    # ---- tables
    def set_embed_tables(self, frame_mod_ab: np.ndarray):
        fm = np.ascontiguousarray(frame_mod_ab, np.uint8)
        assert fm.ndim == 3 and fm.shape[0] == 2 and fm.shape[2] == 101
        self._ck(self.lib.awm_set_embed_tables(self.h, _ptr(fm), ctypes.c_int(fm.shape[1])))

    def set_sync_tables(self, key_slot: int, mode: int, entries: np.ndarray, bit_offsets: np.ndarray):
        e = np.ascontiguousarray(entries, SYNC_ENTRY)
        off = np.ascontiguousarray(bit_offsets, np.int32)
        self._ck(self.lib.awm_set_sync_tables(self.h, ctypes.c_int(key_slot), ctypes.c_int(mode), _ptr(e), ctypes.c_int(len(e)),
                                              _ptr(off), ctypes.c_int(len(off) - 1)))

    def set_mix_tables(self, key_slot: int, entries: np.ndarray, bit_order: np.ndarray, frames_per_bit: int, frames_per_block: int):
        e = np.ascontiguousarray(entries, MIX_ENTRY)
        o = np.ascontiguousarray(bit_order, np.uint16)
        self._ck(self.lib.awm_set_mix_tables(self.h, ctypes.c_int(key_slot), _ptr(e), ctypes.c_int(len(e)), _ptr(o), ctypes.c_int(len(o)),
                                             ctypes.c_int(frames_per_bit), ctypes.c_int(frames_per_block)))

    # ---- PCM
    def pcm_bind(self, pcm, n_frames: int | None = None, channels: int | None = None, pad_start: int = 0, pad_end: int = 0):
        if isinstance(pcm, np.ndarray) and pcm.dtype == np.int16:        # 16 bit PCM: converted on the device
            pcm = np.ascontiguousarray(pcm)
            n_frames, channels = pcm.shape
            self._keep = pcm
            self._ck(self.lib.awm_pcm_bind_s16(self.h, _ptr(pcm), ctypes.c_size_t(n_frames), ctypes.c_int(channels),
                                               ctypes.c_size_t(pad_start), ctypes.c_size_t(pad_end)))
            self.synchronize()
            return
        if isinstance(pcm, np.ndarray):
            pcm = np.ascontiguousarray(pcm, np.float32)
            n_frames, channels = pcm.shape
            self._keep = pcm
        host = isinstance(pcm, np.ndarray)
        self._ck(self.lib.awm_pcm_bind(self.h, _ptr(pcm), ctypes.c_size_t(n_frames), ctypes.c_int(channels),
                                       ctypes.c_size_t(pad_start), ctypes.c_size_t(pad_end)))
        if host or pad_start or pad_end:        # the asynchronous copy reads the caller's array; a device pointer is bound in place
            self.synchronize()

    def pcm_bind_wav(self, data, bits: int, is_float: bool, n_frames: int, channels: int, pad_start: int = 0, pad_end: int = 0, offset: int = 0):
        """bind stored WAV sample bytes (numpy uint8 / bytes from byte `offset` on, or a device pointer), decoded on the device"""
        ptr = self._bytes_ptr(data, offset)
        self._ck(self.lib.awm_pcm_bind_wav(self.h, ptr, WavFormat(bits, int(is_float)), ctypes.c_size_t(n_frames), ctypes.c_int(channels),
                                           ctypes.c_size_t(pad_start), ctypes.c_size_t(pad_end)))
        self.synchronize()

    def pcm_prefetch_wav(self, data, bits: int, is_float: bool, n_frames: int, channels: int, head_frames: int = 0, offset: int = 0):
        """start copying a span of stored WAV samples; its first head_frames frames come from the span prefetched before it and
        `data` (from byte `offset` on) holds the rest.  Bind it with pcm_bind_wav (same data / offset, full n_frames)."""
        ptr = self._bytes_ptr(data, offset)
        self._ck(self.lib.awm_pcm_prefetch_wav(self.h, ptr, WavFormat(bits, int(is_float)), ctypes.c_size_t(n_frames), ctypes.c_int(channels),
                                               ctypes.c_size_t(head_frames)))

    def _bytes_ptr(self, data, offset):
        if isinstance(data, (int, np.integer)):
            return ctypes.c_void_p(int(data) + offset)
        if not isinstance(data, np.ndarray):
            data = np.frombuffer(data, np.uint8)
        data = np.ascontiguousarray(data).view(np.uint8).reshape(-1)
        self._keep_bytes = getattr(self, "_keep_bytes", [])[-3:] + [data]     # the copies read the array asynchronously
        return ctypes.c_void_p(data.ctypes.data + offset)

    def pcm_device(self):
        """(device pointer, frames, channels) of the bound PCM (float32, padding included)"""
        self.lib.awm_pcm_device.restype = ctypes.c_void_p
        n, ch = ctypes.c_size_t(), ctypes.c_int()
        p = self.lib.awm_pcm_device(self.h, ctypes.byref(n), ctypes.byref(ch))
        return int(p or 0), n.value, ch.value

    def copy_to_host(self, dst: np.ndarray, src_ptr: int):
        self._ck(self.lib.awm_copy_to_host(self.h, _ptr(dst), ctypes.c_void_p(src_ptr), ctypes.c_size_t(dst.nbytes)))
        return dst

    # ---- embed
    def embed(self, pcm_in, pcm_out=None, n_frames=None, channels=None, first_frame_number=0, frames_pad_start=250,
              water_delta=0.01, limiter_block=44100, limiter_ceiling=0.99, want_snr=False):
        if isinstance(pcm_in, np.ndarray):
            pcm_in = np.ascontiguousarray(pcm_in, np.float32)
            n_frames, channels = pcm_in.shape
            if pcm_out is None:
                pcm_out = np.empty_like(pcm_in)
        snr = (ctypes.c_double * 2)()
        self._ck(self.lib.awm_embed(self.h, _ptr(pcm_in), _ptr(pcm_out), ctypes.c_size_t(n_frames), ctypes.c_int(channels),
                                    ctypes.c_uint64(first_frame_number), ctypes.c_int(frames_pad_start), ctypes.c_double(water_delta),
                                    ctypes.c_int(limiter_block), ctypes.c_float(limiter_ceiling), snr if want_snr else None))
        return (pcm_out, (snr[0], snr[1])) if want_snr else pcm_out

    # ---- sync
    def sync_approx(self, key_slot=0, mode=MODE_BLOCK, wav_first=0, wav_last=None, water_delta=0.01) -> np.ndarray:
        if wav_last is None:
            wav_last = 0xFFFFFFFFFFFFFFF
        n = ctypes.c_size_t()
        self._ck(self.lib.awm_sync_approx(self.h, ctypes.c_int(key_slot), ctypes.c_int(mode), ctypes.c_uint64(wav_first), ctypes.c_uint64(wav_last),
                                          ctypes.c_double(water_delta), None, ctypes.c_size_t(0), ctypes.byref(n)))
        out = np.zeros(n.value, SEARCH_SCORE)
        if n.value:
            self._ck(self.lib.awm_sync_approx(self.h, ctypes.c_int(key_slot), ctypes.c_int(mode), ctypes.c_uint64(wav_first), ctypes.c_uint64(wav_last),
                                              ctypes.c_double(water_delta), _ptr(out), ctypes.c_size_t(n.value), ctypes.byref(n)))
        return out

    def sync_approx_run(self, key_slot=0, mode=MODE_BLOCK, wav_first=0, wav_last=None, water_delta=0.01) -> int:
        """run the search, keep the scores on the device (for sync_peaks); returns the number of scores"""
        if wav_last is None:
            wav_last = 0xFFFFFFFFFFFFFFF
        n = ctypes.c_size_t()
        self._ck(self.lib.awm_sync_approx(self.h, ctypes.c_int(key_slot), ctypes.c_int(mode), ctypes.c_uint64(wav_first), ctypes.c_uint64(wav_last),
                                          ctypes.c_double(water_delta), None, ctypes.c_size_t(0), ctypes.byref(n)))
        return n.value

    def sync_peaks(self, min_abs_quality: float, max_peaks: int = 65536):
        """local maxima above a floor of the LAST sync_approx call; returns (peaks sorted by index, number found)."""
        out = np.empty(max_peaks, SEARCH_SCORE)
        n = ctypes.c_size_t()
        self._ck(self.lib.awm_sync_peaks(self.h, ctypes.c_double(min_abs_quality), _ptr(out), ctypes.c_size_t(max_peaks), ctypes.byref(n)))
        return out[:min(n.value, max_peaks)].copy(), n.value

    def sync_refine(self, scores: np.ndarray, key_slot=0, mode=MODE_BLOCK, wav_first=0, wav_last=None, water_delta=0.01) -> np.ndarray:
        if wav_last is None:
            wav_last = 0xFFFFFFFFFFFFFFF
        s = np.ascontiguousarray(scores, SEARCH_SCORE).copy()
        self._ck(self.lib.awm_sync_refine(self.h, ctypes.c_int(key_slot), ctypes.c_int(mode), ctypes.c_uint64(wav_first), ctypes.c_uint64(wav_last),
                                          ctypes.c_double(water_delta), _ptr(s), ctypes.c_size_t(len(s))))
        return s

    def sync_refine_offsets(self, scores: np.ndarray, exact: bool, key_slot=0, mode=MODE_BLOCK, wav_first=0, wav_last=None, water_delta=0.01):
        """per-offset qualities of search_refine's 65 fine offsets: sliding-DFT ranking (exact=False) or fresh transforms (exact=True)"""
        if wav_last is None:
            wav_last = 0xFFFFFFFFFFFFFFF
        s = np.ascontiguousarray(scores, SEARCH_SCORE)
        q = np.zeros((len(s), 65), np.float64)
        valid = np.zeros((len(s), 65), np.uint8)
        self._ck(self.lib.awm_sync_refine_offsets(self.h, ctypes.c_int(key_slot), ctypes.c_int(mode), ctypes.c_uint64(wav_first), ctypes.c_uint64(wav_last),
                                                  ctypes.c_double(water_delta), _ptr(s), ctypes.c_size_t(len(s)), ctypes.c_int(1 if exact else 0), _ptr(q), _ptr(valid)))
        return q, valid.astype(bool)

    # ---- decode
    def decode_blocks(self, indices, n_coded: int, key_slot=0):
        idx = np.ascontiguousarray(indices, np.uint64)
        raw = np.zeros((len(idx), n_coded), np.float32)
        valid = np.zeros(len(idx), np.int32)
        self._ck(self.lib.awm_decode_blocks(self.h, ctypes.c_int(key_slot), _ptr(idx), ctypes.c_size_t(len(idx)), _ptr(raw), _ptr(valid)))
        return raw, valid

    def viterbi(self, jobs, block_types, n_msg_bits=128, hard=False):
        """jobs: list of 1-D float arrays (or a 2-D array) of raw soft bits, one per code word (mixed A/B/AB allowed)."""
        jobs = [np.ascontiguousarray(j, np.float32).reshape(-1) for j in jobs]
        bt = np.ascontiguousarray(block_types, np.int32).reshape(-1)
        assert len(jobs) == len(bt)
        for j, t in zip(jobs, bt):
            assert len(j) == (12 if t == BLOCK_AB else 6) * (n_msg_bits + 15)
        raw = np.concatenate(jobs) if jobs else np.zeros(0, np.float32)
        bits = np.zeros((len(jobs), n_msg_bits), np.uint8)
        err = np.zeros(len(jobs), np.float32)
        self._ck(self.lib.awm_viterbi(self.h, _ptr(raw), ctypes.c_size_t(len(jobs)), ctypes.c_int(n_msg_bits), _ptr(bt), ctypes.c_int(1 if hard else 0),
                                      _ptr(bits), _ptr(err)))
        return bits, err

    def resample(self, pcm, ratio: float, n_out: int | None = None, hlen: int = 16, n_frames=None, channels=None, out=None):
        """awm_resample: numpy [n, ch] -> numpy [n_out, ch] (n_out defaults to lrint(n * ratio)); device pointers with sizes given"""
        if isinstance(pcm, np.ndarray):
            pcm = np.ascontiguousarray(pcm, np.float32)
            n_frames, channels = pcm.shape
        if n_out is None:
            n_out = int(np.rint(n_frames * ratio))
        res = np.zeros((n_out, channels), np.float32) if out is None else out
        self._ck(self.lib.awm_resample(self.h, _ptr(pcm), ctypes.c_size_t(n_frames), ctypes.c_int(channels), ctypes.c_double(ratio), ctypes.c_int(hlen),
                                       _ptr(res), ctypes.c_size_t(n_out)))
        return res

    def pcm_push_resampled(self, ratio: float, n_out: int, hlen: int = 16):
        self._ck(self.lib.awm_pcm_push_resampled(self.h, ctypes.c_double(ratio), ctypes.c_int(hlen), ctypes.c_size_t(n_out)))

    def pcm_pop(self):
        self._ck(self.lib.awm_pcm_pop(self.h))

    def speed_scan(self, clip, seconds: float, centers, relative_speeds, key_slot=0, sample_rate=44100, water_delta=0.01,
                   n_frames=None, channels=None) -> np.ndarray:
        """awm_speed_scan: relative_speeds [n_centers][n_rel] -> quality [n_centers][n_rel]"""
        if isinstance(clip, np.ndarray):
            clip = np.ascontiguousarray(clip, np.float32)
            n_frames, channels = clip.shape
        centers = np.ascontiguousarray(centers, np.float64).reshape(-1)
        rel = np.ascontiguousarray(relative_speeds, np.float64).reshape(len(centers), -1)
        out = np.zeros(rel.shape, np.float64)
        self._ck(self.lib.awm_speed_scan(self.h, ctypes.c_int(key_slot), _ptr(clip), ctypes.c_size_t(n_frames), ctypes.c_int(channels), ctypes.c_int(sample_rate),
                                         ctypes.c_double(seconds), _ptr(centers), ctypes.c_int(len(centers)), _ptr(rel), ctypes.c_int(rel.shape[1]),
                                         ctypes.c_double(water_delta), _ptr(out)))
        return out
