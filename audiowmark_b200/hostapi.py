"""ctypes binding of lib/libawm_host.so: the host-side C++ (key tables, `add`, `get`) behind plain C
entry points (audiowmark_b200/host/awm_hostapi.cc).  This is the reference-facing call path the CLI
uses; bench.py's e2e number and the end-to-end parity tests go through it."""
from __future__ import annotations

import ctypes
import json
import os

import numpy as np

from . import capi

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libawm_host.so")
CLI_PATH = os.path.join(_HERE, "bin", "audiowmark")

EXPORTS = ["awmh_set_params", "awmh_frames_per_block", "awmh_n_coded_bits", "awmh_random_u64", "awmh_gen_noise", "awmh_sync_table",
           "awmh_mix_table", "awmh_frame_mod", "awmh_conv_encode", "awmh_add", "awmh_get", "awmh_get_chunk", "awmh_merge_chunks", "awmh_chunk_geometry", "awmh_ctx", "awmh_key_slot", "awmh_stage_select", "awmh_stage_final", "awmh_stage_jobs", "awmh_gpu_launches", "awmh_gpu_stream", "awmh_synchronize", "awmh_profile_enable", "awmh_profile_report", "awmh_shutdown", "awmh_set_speed_params", "awmh_detect_speed", "awmh_resample", "awmh_resample_stream_frames", "awmh_resample_stream_available", "awmh_resampled_add_plan", "awmh_set_short_payload", "awmh_add_s16", "awmh_get_s16", "awmh_short_encode", "awmh_short_decode", "awmh_sync_trace", "awmh_sync_trace_fetch", "awmh_dist_unique_id", "awmh_dist_init", "awmh_balanced_get", "awmh_bg_create", "awmh_bg_destroy", "awmh_bg_stage", "awmh_bg_plan", "awmh_bg_owner", "awmh_add_windowed", "awmh_get_wav", "awmh_wav_decode_host"]

_lib = None


def load():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing: run __graft_entry__.build()" % LIB_PATH)
        capi.load()        # libawm_b200.so first (rpath $ORIGIN also finds it)
        lib = ctypes.CDLL(LIB_PATH)
        lib.awmh_gpu_launches.restype = ctypes.c_uint64
        lib.awmh_gpu_stream.restype = ctypes.c_void_p
        lib.awmh_ctx.restype = ctypes.c_void_p
        _lib = lib
    return _lib


_BUFS = {}


def _outbuf(tag: str, cap: int):
    """persistent ctypes output buffer (create_string_buffer zero-fills: megabytes per call add up in the per-step path)"""
    b = _BUFS.get(tag)
    if b is None or len(b) < cap:
        b = ctypes.create_string_buffer(cap)
        _BUFS[tag] = b
    return b


def _ptr(x):
    if x is None:
        return ctypes.c_void_p(0)
    if isinstance(x, (int, np.integer)):
        return ctypes.c_void_p(int(x))
    assert x.flags["C_CONTIGUOUS"]
    return x.ctypes.data_as(ctypes.c_void_p)


def _key(key) -> bytes:
    k = bytes(key) if key is not None else bytes(16)
    assert len(k) == 16
    return k


_PARAMS = {"sync_threshold2": 0.35, "n_best": 8, "water_delta": 0.01}


def get_param(name):
    return _PARAMS[name]


def set_params(water_delta=0.01, frames_per_bit=2, mix=True, hard=False, sync_threshold2=0.35, n_best=8, chunk_size_min=30.0,
               test_no_limiter=False, test_no_sync=False, gpu_device=0, quiet=True):
    _PARAMS.update(sync_threshold2=sync_threshold2, n_best=n_best, water_delta=water_delta)
    load().awmh_set_params(ctypes.c_double(water_delta), ctypes.c_int(frames_per_bit), ctypes.c_int(mix), ctypes.c_int(hard),
                           ctypes.c_double(sync_threshold2), ctypes.c_int(n_best), ctypes.c_double(chunk_size_min),
                           ctypes.c_int(test_no_limiter), ctypes.c_int(test_no_sync), ctypes.c_int(gpu_device), ctypes.c_int(quiet))


def frames_per_block() -> int:
    return load().awmh_frames_per_block()


def n_coded_bits() -> int:
    return load().awmh_n_coded_bits()


def random_u64(key, seed: int, stream: int, n: int) -> np.ndarray:
    out = np.zeros(n, np.uint64)
    load().awmh_random_u64(_key(key), ctypes.c_uint64(seed), ctypes.c_int(stream), _ptr(out), ctypes.c_int(n))
    return out


def gen_noise(key, n_values: int) -> np.ndarray:
    out = np.zeros(n_values, np.float32)
    load().awmh_gen_noise(_key(key), _ptr(out), ctypes.c_size_t(n_values))
    return out


def sync_table(key, mode: int):
    ent = np.zeros(4096, capi.SYNC_ENTRY)
    off = np.zeros(7, np.int32)
    n = load().awmh_sync_table(_key(key), ctypes.c_int(mode), _ptr(ent), ctypes.c_int(len(ent)), _ptr(off))
    assert n > 0
    return ent[:n].copy(), off


def mix_table(key):
    ent = np.zeros(200000, capi.MIX_ENTRY)
    order = np.zeros(8192, np.uint16)
    n = load().awmh_mix_table(_key(key), _ptr(ent), ctypes.c_int(len(ent)), _ptr(order), ctypes.c_int(len(order)))
    assert n > 0
    return ent[:n].copy(), order[:n_coded_bits()].copy()


def frame_mod(key, payload_hex: str) -> np.ndarray:
    fpb = frames_per_block()
    out = np.zeros((2, fpb, 101), np.uint8)
    n = load().awmh_frame_mod(_key(key), payload_hex.encode(), _ptr(out), ctypes.c_size_t(out.size))
    assert n == out.size
    return out


def conv_encode(block_type: int, bits) -> np.ndarray:
    b = np.ascontiguousarray(bits, np.uint8)
    out = np.zeros((len(b) + 15) * 12, np.uint8)
    n = load().awmh_conv_encode(ctypes.c_int(block_type), _ptr(b), ctypes.c_int(len(b)), _ptr(out), ctypes.c_int(len(out)))
    return out[:n].copy()


def short_encode(bits) -> np.ndarray:
    """block code of the current --short mode: k message bits -> n code bits"""
    b = np.ascontiguousarray(bits, np.uint8)
    out = np.zeros(128, np.uint8)
    n = load().awmh_short_encode(_ptr(b), ctypes.c_int(len(b)), _ptr(out), ctypes.c_int(len(out)))
    if n < 0:
        raise ValueError("short payload mode is off or the message length does not match")
    return out[:n].copy()


def short_decode(coded) -> np.ndarray:
    """n code bits -> k message bits; empty if no code word matches"""
    c = np.ascontiguousarray(coded, np.uint8)
    out = np.zeros(32, np.uint8)
    n = load().awmh_short_decode(_ptr(c), ctypes.c_int(len(c)), _ptr(out), ctypes.c_int(len(out)))
    if n < 0:
        raise ValueError("short payload mode is off or the code length does not match")
    return out[:n].copy()


def add(pcm_in, payload_hex: str, key=None, pcm_out=None, n_frames=None, channels=None, sample_rate=44100, want_stats=False, first_frame_number=0):
    """add_stream_watermark on a buffer: numpy arrays (host) or device pointers (ints)."""
    if isinstance(pcm_in, np.ndarray):
        pcm_in = np.ascontiguousarray(pcm_in, np.float32)
        n_frames, channels = pcm_in.shape
        if pcm_out is None:
            pcm_out = np.empty_like(pcm_in)
    blocks, snr = ctypes.c_int(), ctypes.c_double()
    rc = load().awmh_add(_key(key), _ptr(pcm_in), _ptr(pcm_out), ctypes.c_size_t(n_frames), ctypes.c_int(channels), ctypes.c_int(sample_rate),
                         payload_hex.encode(), ctypes.byref(blocks) if want_stats else None, ctypes.byref(snr) if want_stats else None,
                         ctypes.c_uint64(first_frame_number))
    if rc:
        raise RuntimeError("awmh_add failed (rc=%d); see stderr" % rc)
    return (pcm_out, blocks.value, snr.value) if want_stats else pcm_out


def add_windowed(pcm_in: np.ndarray, payload_hex: str, key=None, zero_frames=0, window_frames=0, sample_rate=44100):
    """the bounded-memory loop of `audiowmark add` (add_watermark_windowed) on a host buffer -> (output, data blocks, snr dB)"""
    pcm_in = np.ascontiguousarray(pcm_in, np.float32)
    out = np.empty_like(pcm_in)
    blocks, snr = ctypes.c_int(), ctypes.c_double()
    rc = load().awmh_add_windowed(_key(key), _ptr(pcm_in), _ptr(out), ctypes.c_size_t(pcm_in.shape[0]), ctypes.c_int(pcm_in.shape[1]), ctypes.c_int(sample_rate),
                                  payload_hex.encode(), ctypes.c_size_t(zero_frames), ctypes.c_size_t(window_frames), ctypes.byref(blocks), ctypes.byref(snr))
    if rc:
        raise RuntimeError("awmh_add_windowed failed (rc=%d); see stderr" % rc)
    return out, blocks.value, snr.value


def get(pcm, keys=None, names=None, n_frames=None, channels=None, sample_rate=44100, parse=True):
    """get_watermark on a buffer -> the --json document (dict) of the run."""
    keys = keys or [bytes(16)]
    names = names or [""] * len(keys)
    if isinstance(pcm, np.ndarray):
        pcm = np.ascontiguousarray(pcm, np.float32)
        n_frames, channels = pcm.shape
    kb = b"".join(_key(k) for k in keys)
    name_arr = (ctypes.c_char_p * len(keys))(*[n.encode() for n in names])
    cap = 1 << 22
    buf = _outbuf("get", cap)
    n_pat = ctypes.c_int()
    rc = load().awmh_get(kb, name_arr, ctypes.c_int(len(keys)), _ptr(pcm), ctypes.c_size_t(n_frames), ctypes.c_int(channels),
                         ctypes.c_int(sample_rate), buf, ctypes.c_size_t(cap), ctypes.byref(n_pat))
    if rc:
        raise RuntimeError("awmh_get failed (rc=%d); see stderr" % rc)
    text = buf.value.decode()
    return json.loads(text) if parse else text


def get_wav_bytes(data, channels, bits, is_float=False, sample_rate=44100, keys=None, names=None, chunk_buffer=None, parse=True):
    """`get` on the stored sample bytes of a WAV file (bytes or numpy; 8 bit unsigned, 16/24/32 bit signed, 32/64 bit float, little
    endian) -> the --json document.  At 44.1 kHz this is the CLI's streamed loader over a memory buffer: chunks are read into two
    page-locked buffers and decoded on the device.  chunk_buffer: frames handed out per read of the buffer, as a pipe delivers short
    reads (None: a whole chunk per read); it does not change the result."""
    keys = keys or [bytes(16)]
    names = names or [""] * len(keys)
    if not isinstance(data, np.ndarray):
        data = np.frombuffer(data, np.uint8)
    data = np.ascontiguousarray(data).view(np.uint8).reshape(-1)
    kb = b"".join(_key(k) for k in keys)
    name_arr = (ctypes.c_char_p * len(keys))(*[n.encode() for n in names])
    cap = 1 << 22
    buf = _outbuf("get", cap)
    n_pat = ctypes.c_int()
    rc = load().awmh_get_wav(kb, name_arr, ctypes.c_int(len(keys)), _ptr(data), ctypes.c_size_t(data.nbytes), ctypes.c_int(channels),
                             ctypes.c_int(bits), ctypes.c_int(int(is_float)), ctypes.c_int(sample_rate), ctypes.c_size_t(chunk_buffer or 0),
                             buf, ctypes.c_size_t(cap), ctypes.byref(n_pat))
    if rc:
        raise RuntimeError("awmh_get_wav failed (rc=%d); see stderr" % rc)
    text = buf.value.decode()
    return json.loads(text) if parse else text


def wav_decode_host(data, bits, is_float=False) -> np.ndarray:
    """test aid: the host's RawConverter::from_raw of stored WAV sample bytes -> float32 (one value per sample)"""
    if not isinstance(data, np.ndarray):
        data = np.frombuffer(data, np.uint8)
    data = np.ascontiguousarray(data).view(np.uint8).reshape(-1)
    n = data.nbytes // (bits // 8)
    out = np.empty(n, np.float32)
    if load().awmh_wav_decode_host(_ptr(data), ctypes.c_size_t(n), ctypes.c_int(bits), ctypes.c_int(int(is_float)), _ptr(out)):
        raise ValueError("unsupported sample format: %d bit %s" % (bits, "float" if is_float else "integer"))
    return out


def sync_trace(on=True):
    """test aid: record what every SyncFinder::search call returns from now on (see sync_trace_fetch)"""
    load().awmh_sync_trace(ctypes.c_int(1 if on else 0))


def sync_trace_fetch():
    """-> list of searches in call order: {"mode": "BLOCK"|"CLIP", "n_frames": int, "scores": [[index, quality, "A"|"B"], ...]}
    (the format of oracle/ref_shims/sync_dump.cc's print-out as tests/golden/make_golden_large.py stores it)"""
    cap = 1 << 16
    rows = np.zeros((cap, 5), np.float64)
    n = ctypes.c_size_t()
    if load().awmh_sync_trace_fetch(_ptr(rows), ctypes.c_size_t(cap), ctypes.byref(n)):
        raise RuntimeError("sync trace longer than %d rows" % cap)
    out = []
    for r in rows[:n.value]:
        if r[3] < 0:
            out.append({"mode": "CLIP" if r[1] else "BLOCK", "n_frames": int(r[2]), "scores": []})
        else:
            out[-1]["scores"].append([int(r[1]), float(r[2]), "B" if r[3] else "A"])
    return out


def set_short_payload(bits=0):
    """--short <bits> (12, 16, 20); 0 = normal 128 bit payload"""
    if load().awmh_set_short_payload(ctypes.c_int(bits)) < 0:
        raise ValueError("unsupported short payload size %d" % bits)


def set_speed_params(detect_speed=False, detect_speed_patient=False, try_speed=-1.0, test_speed=-1.0):
    """--detect-speed / --detect-speed-patient / --try-speed / --test-speed of `audiowmark get`"""
    load().awmh_set_speed_params(ctypes.c_int(int(detect_speed)), ctypes.c_int(int(detect_speed_patient)), ctypes.c_double(try_speed),
                                 ctypes.c_double(test_speed))


def detect_speed(pcm, key=None, n_frames=None, channels=None, sample_rate=44100):
    """detect_speed for one key on one chunk -> (speed, quality, accepted)"""
    if isinstance(pcm, np.ndarray):
        pcm = np.ascontiguousarray(pcm, np.float32)
        n_frames, channels = pcm.shape
    sp, q, acc = ctypes.c_double(), ctypes.c_double(), ctypes.c_int()
    rc = load().awmh_detect_speed(_key(key or bytes(16)), _ptr(pcm), ctypes.c_size_t(n_frames), ctypes.c_int(channels), ctypes.c_int(sample_rate),
                                  ctypes.byref(sp), ctypes.byref(q), ctypes.byref(acc))
    if rc:
        raise RuntimeError("awmh_detect_speed failed (rc=%d); see stderr" % rc)
    return sp.value, q.value, bool(acc.value)


def resample(pcm, ratio, n_out=None, out=None, n_frames=None, channels=None):
    """resample_ratio: numpy in -> numpy out, or device pointers with n_frames / channels / n_out given"""
    if isinstance(pcm, np.ndarray):
        pcm = np.ascontiguousarray(pcm, np.float32)
        n_frames, channels = pcm.shape
    if n_out is None:
        n_out = int(np.rint(n_frames * ratio))
    res = out
    if out is None:
        res = np.zeros((n_out, channels), np.float32)
    rc = load().awmh_resample(_ptr(pcm), ctypes.c_size_t(n_frames), ctypes.c_int(channels), ctypes.c_double(ratio), _ptr(res), ctypes.c_size_t(n_out))
    if rc:
        raise RuntimeError("awmh_resample failed (rc=%d); see stderr" % rc)
    return res


def resample_stream_frames(n_in, ratio):
    L = load()
    L.awmh_resample_stream_frames.restype = ctypes.c_uint64
    return int(L.awmh_resample_stream_frames(ctypes.c_uint64(n_in), ctypes.c_double(ratio)))


def resample_stream_available(fed, ratio):
    L = load()
    L.awmh_resample_stream_available.restype = ctypes.c_uint64
    return int(L.awmh_resample_stream_available(ctypes.c_uint64(fed), ctypes.c_double(ratio)))


def resampled_add_plan(n_frames, sample_rate):
    """(frames through the mixer, WatermarkGen::run calls) of `add` at a sample rate other than 44.1 kHz"""
    e, r = ctypes.c_uint64(), ctypes.c_uint64()
    load().awmh_resampled_add_plan(ctypes.c_uint64(n_frames), ctypes.c_int(sample_rate), ctypes.byref(e), ctypes.byref(r))
    return e.value, r.value


def add_s16(pcm_in, payload_hex: str, key=None, pcm_out=None, sample_rate=44100, want_stats=False, first_frame_number=0):
    """`add` between 16 bit PCM host buffers (int16 numpy [n, ch]): the int <-> float conversions run on the device"""
    pcm_in = np.ascontiguousarray(pcm_in, np.int16)
    n_frames, channels = pcm_in.shape
    if pcm_out is None:
        pcm_out = np.empty_like(pcm_in)
    blocks, snr = ctypes.c_int(), ctypes.c_double()
    rc = load().awmh_add_s16(_key(key), _ptr(pcm_in), _ptr(pcm_out), ctypes.c_size_t(n_frames), ctypes.c_int(channels), ctypes.c_int(sample_rate),
                             payload_hex.encode(), ctypes.byref(blocks) if want_stats else None, ctypes.byref(snr) if want_stats else None,
                             ctypes.c_uint64(first_frame_number))
    if rc:
        raise RuntimeError("awmh_add_s16 failed (rc=%d); see stderr" % rc)
    return (pcm_out, blocks.value, snr.value) if want_stats else pcm_out


def get_s16(pcm, keys=None, names=None, sample_rate=44100, parse=True):
    """`get` on a 16 bit PCM host buffer (int16 numpy [n, ch]) -> the --json document"""
    keys = keys or [bytes(16)]
    names = names or [""] * len(keys)
    pcm = np.ascontiguousarray(pcm, np.int16)
    n_frames, channels = pcm.shape
    kb = b"".join(_key(k) for k in keys)
    name_arr = (ctypes.c_char_p * len(keys))(*[n.encode() for n in names])
    cap = 1 << 22
    buf = _outbuf("get", cap)
    n_pat = ctypes.c_int()
    rc = load().awmh_get_s16(kb, name_arr, ctypes.c_int(len(keys)), _ptr(pcm), ctypes.c_size_t(n_frames), ctypes.c_int(channels),
                             ctypes.c_int(sample_rate), buf, ctypes.c_size_t(cap), ctypes.byref(n_pat))
    if rc:
        raise RuntimeError("awmh_get_s16 failed (rc=%d); see stderr" % rc)
    text = buf.value.decode()
    return json.loads(text) if parse else text


def chunk_geometry(sample_rate=44100):
    """(max_frames, overlap_frames) of the reference's WavChunkLoader for the current --chunk-size."""
    m, o = ctypes.c_uint64(), ctypes.c_uint64()
    load().awmh_chunk_geometry(ctypes.c_int(sample_rate), ctypes.byref(m), ctypes.byref(o))
    return m.value, o.value


def get_chunk(pcm, first_chunk: bool, keys=None, names=None, n_frames=None, channels=None, sample_rate=44100) -> bytes:
    """decode one chunk; returns the chunk's pattern records (bytes) for merge_chunks."""
    keys = keys or [bytes(16)]
    names = names or [""] * len(keys)
    if isinstance(pcm, np.ndarray):
        pcm = np.ascontiguousarray(pcm, np.float32)
        n_frames, channels = pcm.shape
    kb = b"".join(_key(k) for k in keys)
    name_arr = (ctypes.c_char_p * len(keys))(*[n.encode() for n in names])
    cap = 1 << 20
    buf = ctypes.create_string_buffer(cap)
    blen = ctypes.c_size_t()
    rc = load().awmh_get_chunk(kb, name_arr, ctypes.c_int(len(keys)), _ptr(pcm), ctypes.c_size_t(n_frames), ctypes.c_int(channels),
                               ctypes.c_int(sample_rate), ctypes.c_int(1 if first_chunk else 0), buf, ctypes.c_size_t(cap), ctypes.byref(blen))
    if rc:
        raise RuntimeError("awmh_get_chunk failed (rc=%d); see stderr" % rc)
    return ctypes.string_at(buf, blen.value)


def merge_chunks(blobs, time_offsets, total_seconds: float, keys=None, names=None) -> dict:
    """ResultSet::merge in chunk order + sort -> the --json document."""
    keys = keys or [bytes(16)]
    names = names or [""] * len(keys)
    kb = b"".join(_key(k) for k in keys)
    name_arr = (ctypes.c_char_p * len(keys))(*[n.encode() for n in names])
    n = len(blobs)
    bufs = [(ctypes.c_ubyte * max(len(b), 1)).from_buffer_copy(b if b else b"\0") for b in blobs]
    ptrs = (ctypes.POINTER(ctypes.c_ubyte) * n)(*[ctypes.cast(b, ctypes.POINTER(ctypes.c_ubyte)) for b in bufs])
    lens = (ctypes.c_size_t * n)(*[len(b) for b in blobs])
    offs = (ctypes.c_double * n)(*time_offsets)
    cap = 1 << 22
    out = _outbuf("merge", cap)
    rc = load().awmh_merge_chunks(kb, name_arr, ctypes.c_int(len(keys)), ptrs, lens, offs, ctypes.c_int(n), ctypes.c_double(total_seconds),
                                  out, ctypes.c_size_t(cap))
    if rc:
        raise RuntimeError("awmh_merge_chunks failed (rc=%d)" % rc)
    return json.loads(out.value.decode())


# ---- sharded get: one long stream over several GPUs, one process per GPU (host/awm_balanced.hh) -----------------------------

def dist_unique_id() -> bytes:
    """NCCL unique id of a new job (rank 0 creates it, the launcher hands it to every rank)"""
    buf = ctypes.create_string_buffer(128)
    if load().awmh_dist_unique_id(buf):
        raise RuntimeError("NCCL is not available")
    return buf.raw


def dist_init(rank: int, world: int, unique_id: bytes):
    """join the job's NCCL communicator (exchanges of the sharded get run on the context stream)"""
    if load().awmh_dist_init(ctypes.c_int(rank), ctypes.c_int(world), ctypes.c_char_p(unique_id)):
        raise RuntimeError("awmh_dist_init failed; see stderr")


def dist_init_from_torch():
    """the usual launcher: torch.distributed is up (torchrun); rank 0's id is broadcast through it"""
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", torch.cuda.current_device())
    t = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        t.copy_(torch.frombuffer(bytearray(dist_unique_id()), dtype=torch.uint8))
    dist.broadcast(t, 0)
    dist_init(rank, world, bytes(t.cpu().numpy().tobytes()))


def balanced_get(pcm, pcm_start: int, n_total: int, key=None, n_frames=None, channels=None, sample_rate=44100, parse=True):
    """this rank's part of the stream (numpy float32 / int16 [n, ch], or a float32 device pointer) -> the --json document on rank 0
    (parse=False: its text, as `audiowmark get --json` writes it), None on the other ranks"""
    is_s16 = 0
    if isinstance(pcm, np.ndarray):
        if pcm.dtype == np.int16:
            pcm, is_s16 = np.ascontiguousarray(pcm), 1
        else:
            pcm = np.ascontiguousarray(pcm, np.float32)
        n_frames, channels = pcm.shape
    cap = 1 << 22
    buf = _outbuf("get", cap)
    n_pat = ctypes.c_int()
    rc = load().awmh_balanced_get(_key(key), _ptr(pcm), ctypes.c_int(is_s16), ctypes.c_uint64(pcm_start), ctypes.c_uint64(n_frames), ctypes.c_uint64(n_total),
                                  ctypes.c_int(channels), ctypes.c_int(sample_rate), buf, ctypes.c_size_t(cap), ctypes.byref(n_pat))
    if rc:
        raise RuntimeError("awmh_balanced_get failed (rc=%d); see stderr" % rc)
    if n_pat.value < 0:
        return None
    text = buf.value.decode()
    return json.loads(text) if parse else text


class BalancedStages:
    """one rank of the sharded get with the stages callable one by one (tests run several ranks in one process on one GPU)"""

    def __init__(self, rank, world, n_total, pcm_device_ptr: int, pcm_frames: int, channels: int, pcm_start, key=None, sample_rate=44100):
        """pcm_device_ptr: float32 [pcm_frames, channels] in device memory that stays valid while the object lives (several ranks in
        one process share the context, so each needs its own device copy -- a host buffer would land in the context's single
        upload buffer)"""
        self.n_total = n_total
        L = load()
        L.awmh_bg_create.restype = ctypes.c_void_p
        self.h = L.awmh_bg_create(_key(key), ctypes.c_int(rank), ctypes.c_int(world), ctypes.c_void_p(pcm_device_ptr), ctypes.c_uint64(pcm_start),
                                  ctypes.c_uint64(pcm_frames), ctypes.c_uint64(n_total), ctypes.c_int(channels), ctypes.c_int(sample_rate))
        if not self.h:
            raise RuntimeError("awmh_bg_create failed; see stderr")

    def stage(self, number: int, payloads=()) -> bytes:
        n = len(payloads)
        arr = (ctypes.c_char_p * max(n, 1))(*[bytes(p) for p in payloads]) if n else None
        lens = (ctypes.c_size_t * max(n, 1))(*[len(p) for p in payloads])
        cap = 1 << 24
        out = _outbuf("bg", cap)
        out_len = ctypes.c_size_t()
        rc = load().awmh_bg_stage(ctypes.c_void_p(self.h), ctypes.c_int(number), arr, lens, ctypes.c_int(n), ctypes.c_uint64(self.n_total), out, ctypes.c_size_t(cap),
                                  ctypes.byref(out_len))
        if rc:
            raise RuntimeError("awmh_bg_stage %d failed (rc=%d)" % (number, rc))
        return out.raw[:out_len.value]

    def close(self):
        if self.h:
            load().awmh_bg_destroy(ctypes.c_void_p(self.h))
            self.h = None


def balanced_plan(n_total: int, rank: int, world: int, sample_rate=44100):
    """-> (chunks [(first, count, time offset)], slices [(chunk, sa, sb, a, b, lo, hi)]) as the C++ driver computes them"""
    chunks = np.zeros((64, 3), np.float64)
    slices = np.zeros((64, 7), np.int64)
    nc, ns = ctypes.c_int(), ctypes.c_int()
    load().awmh_bg_plan(ctypes.c_uint64(n_total), ctypes.c_int(sample_rate), ctypes.c_int(rank), ctypes.c_int(world), _ptr(chunks), ctypes.c_int(64), ctypes.byref(nc),
                        _ptr(slices), ctypes.c_int(64), ctypes.byref(ns))
    return [(int(a), int(b), float(t)) for a, b, t in chunks[:nc.value]], [tuple(int(v) for v in row) for row in slices[:ns.value]]


def balanced_owner(n_total: int, world: int, chunk: int, index: int, sample_rate=44100) -> int:
    return load().awmh_bg_owner(ctypes.c_uint64(n_total), ctypes.c_int(sample_rate), ctypes.c_int(world), ctypes.c_int(chunk), ctypes.c_uint64(index))


def engine_ctx() -> int:
    """awm_ctx* of the host library's GPU context (creates it; raises without a CUDA device)"""
    h = load().awmh_ctx()
    if not h:
        raise RuntimeError("no GPU context: a CUDA device is required, there is no CPU fallback")
    return int(h)


def key_slot(key=None) -> int:
    s = load().awmh_key_slot(_key(key))
    if s < 0:
        raise RuntimeError("key table upload failed")
    return s


def stage_select(peaks: np.ndarray, floor_q: float, clip_mode=False):
    pk = np.ascontiguousarray(peaks, capi.SEARCH_SCORE)
    out = np.zeros(max(len(pk), 1), capi.SEARCH_SCORE)
    n, complete = ctypes.c_size_t(), ctypes.c_int()
    rc = load().awmh_stage_select(_ptr(pk), ctypes.c_size_t(len(pk)), ctypes.c_double(floor_q), ctypes.c_int(1 if clip_mode else 0),
                                  _ptr(out), ctypes.c_size_t(len(out)), ctypes.byref(n), ctypes.byref(complete))
    if rc:
        raise RuntimeError("awmh_stage_select failed (%d)" % rc)
    return out[:n.value].copy(), bool(complete.value)


def stage_final(refined: np.ndarray):
    r = np.ascontiguousarray(refined, capi.SEARCH_SCORE)
    idx, q, bt = np.zeros(len(r), np.uint64), np.zeros(len(r), np.float64), np.zeros(len(r), np.int32)
    n = ctypes.c_size_t()
    load().awmh_stage_final(_ptr(r), ctypes.c_size_t(len(r)), _ptr(idx), _ptr(q), _ptr(bt), ctypes.byref(n))
    return idx[:n.value].copy(), q[:n.value].copy(), bt[:n.value].copy()


def stage_jobs(key, index, quality, btype, raw, valid, sample_rate=44100):
    """Viterbi jobs of one chunk: list of (code_type, pattern_type, score_btype, time, index, quality, soft float32[])"""
    import struct
    idx, q, bt = (np.ascontiguousarray(index, np.uint64), np.ascontiguousarray(quality, np.float64), np.ascontiguousarray(btype, np.int32))
    raw = np.ascontiguousarray(raw, np.float32)
    valid = np.ascontiguousarray(valid, np.int32)
    cap = 64 + (len(idx) * 3 + 2) * (36 + raw.shape[1] * 8) if len(idx) else 64
    buf = _outbuf("jobs", cap)
    blen, nj = ctypes.c_size_t(), ctypes.c_int()
    rc = load().awmh_stage_jobs(_key(key), _ptr(idx), _ptr(q), _ptr(bt), ctypes.c_size_t(len(idx)), _ptr(raw), _ptr(valid), ctypes.c_int(sample_rate),
                                buf, ctypes.c_size_t(cap), ctypes.byref(blen), ctypes.byref(nj))
    if rc:
        raise RuntimeError("awmh_stage_jobs failed (%d)" % rc)
    data = ctypes.string_at(buf, blen.value)
    out, pos = [], 0
    for _ in range(nj.value):
        ct, pt, sbt, _pad, time, index_, quality_, n_soft = struct.unpack_from("<BBBBdQdI", data, pos)
        pos += 32
        soft = np.frombuffer(data, np.float32, n_soft, pos).copy()
        pos += 4 * n_soft
        out.append((ct, pt, sbt, time, index_, quality_, soft))
    return out


def gpu_launches() -> int:
    return int(load().awmh_gpu_launches())


def gpu_stream() -> int:
    return int(load().awmh_gpu_stream() or 0)


def synchronize():
    """wait for the context stream (calls with DEVICE pointers are asynchronous)."""
    if load().awmh_synchronize():
        raise RuntimeError("no GPU context")


def profile_enable(on=True):
    if load().awmh_profile_enable(ctypes.c_int(1 if on else 0)):
        raise RuntimeError("no GPU context")


def profile_report() -> dict:
    buf = ctypes.create_string_buffer(1 << 16)
    if load().awmh_profile_report(buf, ctypes.c_size_t(len(buf))):
        raise RuntimeError("awmh_profile_report failed")
    return json.loads(buf.value.decode())


def shutdown():
    if _lib is not None:
        _lib.awmh_shutdown()
