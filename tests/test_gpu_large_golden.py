"""GPU, BASELINE.json's configs 2-4 at their stated sizes and the digital-silence cases, against documents and sync positions
printed by the UNMODIFIED reference (tests/golden/golden_large.json, made by tests/golden/make_golden_large.py from
oracle/_ref/audiowmark and oracle/_ref/sync_dump):

  config 2   1 h stereo add + get: all 108 patterns of the reference's --json document, the 75 sync scores of its three chunks
  config 3   30 s clip cut from the 1 h output by test-clip (seed 0): clip decoder, 8 sync scores
  config 4   --detect-speed on 10 min stereo at speeds 0.9 / 0.9764 / 1.01 / 1.1 (the edges of the +-10 % scan range included)
  silence    170 s of zeros; 60 s of watermarked noise followed by 60 s of zeros
  music      music-like (pink noise + steady tones), a -6 dBFS tone over a 1 LSB floor, -60 dBFS music, clipped music with DC,
             one-sided stereo (R silent, R at -50 dB, R = L, R = -L), mono and 3 channels: 130 s (clip decoder runs too) or 170 s
             (three sync blocks); 10 min stereo music, also watermarked with two named keys

The inputs are regenerated here from seeds with the oracle (keyed noise generator, bit exact embedder, resampler) and checked
against the SHA-256 of what the reference binary read -- the GPU `get` sees byte for byte the reference's input.

Bars: bits, block type, position, key and ORDER of every pattern identical; sync indices IDENTICAL (north_star: "bit-exact ...
sync positions") -- a deviation of one sync_search_fine step (8 samples) is counted separately and must not occur on these
cases; quality within 2e-4 / error within 2e-3 of the printed values; detected speed within 2e-6."""
import hashlib
import json
import os

import numpy as np
import pytest

import awm_oracle as O
import awm_testlib as T
from audiowmark_b200 import hostapi as H

pytestmark = pytest.mark.gpu
G = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_large.json")))
RATE = 44100
PAYLOAD = "f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0"


def sha16(x16):
    return hashlib.sha256(np.ascontiguousarray(x16).tobytes()).hexdigest()


def compare_docs(got, want, q_tol=2e-4, e_tol=2e-3, thr=0.35):
    """every pattern, fillers (n-best entries below the sync threshold: decoded noise) included -> number of real patterns"""
    assert got["length"] == want["length"]
    gm, wm = got["matches"], want["matches"]
    assert len(gm) == len(wm), (len(gm), len(wm))
    for i, (g, w) in enumerate(zip(gm, wm)):
        assert (g["key"], g["pos"], g["bits"], g["type"]) == (w["key"], w["pos"], w["bits"], w["type"]), (i, g, w)
        assert abs(g["quality"] - w["quality"]) < q_tol and abs(g["error"] - w["error"]) < e_tol and abs(g["rating"] - w["rating"]) < 10 * q_tol, (i, g, w)
        assert abs(g["speed"] - w["speed"]) < 2e-6, (i, g, w)
    return sum(1 for m in wm if m["quality"] > thr)


def compare_sync(got, want, q_tol=2e-4):
    """sync positions of every SyncFinder::search call -> (scores compared, scores that are one fine step off)"""
    assert [(s["mode"], s["n_frames"], len(s["scores"])) for s in got] == [(s["mode"], s["n_frames"], len(s["scores"])) for s in want]
    n = off_by_step = 0
    for sg, sw in zip(got, want):
        for (gi, gq, gt), (wi, wq, wt) in zip(sg["scores"], sw["scores"]):
            n += 1
            assert gt == wt and abs(gq - wq) < q_tol, (sg["mode"], gi, gq, gt, wi, wq, wt)
            if gi != wi:
                assert abs(gi - wi) <= 8, (sg["mode"], gi, wi)
                off_by_step += 1
    return n, off_by_step


def get_with_trace(x, **kw):
    H.set_params()
    H.sync_trace(True)
    try:
        doc = H.get(x, **kw)
        return doc, H.sync_trace_fetch()
    finally:
        H.sync_trace(False)


def test_silence170_vs_reference():
    g = G["silence170"]
    doc, trace = get_with_trace(np.zeros((g["seconds"] * RATE, 2), np.float32))
    assert compare_docs(doc, g["json"], q_tol=1e-9, e_tol=1e-6) == 0
    assert [m["error"] for m in doc["matches"]] == [-0.001166] * 4          # -1 / 858: no path survives NaN soft bits
    assert compare_sync(trace, g["sync"], q_tol=1e-12) == (8, 0)


def test_noise_then_silence_vs_reference():
    g = G["noise60_silence60"]
    x = O.int16_to_float(O.quantize_sndfile16(T.noise(60.0, 2, seed=g["noise_seed"])))
    y16 = O.quantize_sndfile16(O.embed(x, O.Key(), PAYLOAD, O.Params()).samples)
    assert sha16(y16) == g["wm_sha256"]
    ns = np.concatenate([y16, np.zeros((60 * RATE, 2), np.int16)])
    assert sha16(ns) == g["input_sha256"]
    doc, trace = get_with_trace(O.int16_to_float(ns))
    assert compare_docs(doc, g["json"]) == 2
    assert compare_sync(trace, g["sync"]) == (24, 0)


@pytest.fixture(scope="module")
def hour16():
    """the reference's 1 h output file, regenerated: keyed noise (test-gen-noise) on the 16 bit grid, embedded by the oracle"""
    g = G["hour"]
    x16 = O.quantize_sndfile16(O.gen_noise(3600))
    assert sha16(x16) == g["input_sha256"]
    y16 = O.quantize_sndfile16(O.embed(O.int16_to_float(x16), O.Key(), PAYLOAD, O.Params()).samples)
    del x16
    assert sha16(y16) == g["output_sha256"]
    return y16


def test_hour_vs_reference(hour16):
    g = G["hour"]
    doc, trace = get_with_trace(O.int16_to_float(hour16))
    n_real = compare_docs(doc, g["json"])
    assert len(doc["matches"]) == 108 and n_real == 104                       # 4 fillers below the sync threshold
    assert sum(m["bits"] == PAYLOAD for m in doc["matches"]) == 104           # cmp: match_count 104 108
    assert compare_sync(trace, g["sync"]) == (75, 0)
    # the 16 bit entry point (what bench.py's e2e leg calls) gives the same document
    assert H.get_s16(np.ascontiguousarray(hour16)) == doc


def test_clip30_vs_reference(hour16):
    g = G["clip30"]
    assert sha16(hour16[:140 * RATE]) == G["hour"]["output_head140_sha256"]
    c16 = hour16[g["start_frame"]: g["start_frame"] + g["n_frames"]]
    assert sha16(c16) == g["input_sha256"]
    doc, trace = get_with_trace(O.int16_to_float(c16))
    assert compare_docs(doc, g["json"]) == 1
    assert doc["matches"][0]["bits"] == PAYLOAD and doc["matches"][0]["type"] == "CLIP-B"
    assert compare_sync(trace, g["sync"]) == (8, 0)


@pytest.mark.parametrize("idx", range(4))
def test_detect_speed_10min_vs_reference(hour16, idx):
    g = G["speed600"]["cases"][idx]
    assert sha16(hour16[:600 * RATE]) == G["hour"]["output_head600_sha256"]
    m10 = O.int16_to_float(hour16[:600 * RATE])
    s16 = O.quantize_sndfile16(O.resample_ratio(m10, 1 / T.cli_float(g["speed"])))      # test-change-speed, saved as 16 bit
    assert len(s16) == g["n_frames"] and sha16(s16) == g["input_sha256"]
    H.set_params()
    H.set_speed_params(detect_speed=True)
    try:
        doc = H.get(O.int16_to_float(s16))
    finally:
        H.set_speed_params()
    n_real = compare_docs(doc, g["json"])
    speed_hits = [m for m in doc["matches"] if m["type"].endswith("-SPEED") and m["bits"] == PAYLOAD]
    assert n_real >= 10 and len(speed_hits) >= 10
    assert all(abs(m["speed"] - g["speed"]) < 1e-4 for m in speed_hits)


# ---- tonal, quiet, clipped, one-sided stereo, mono and 3-channel inputs (tests/awm_testlib.py signals), watermarked by the reference
MUSIC_CASES = ["music130", "tone170", "quiet130", "dc_clip130", "r_zero130", "r_m50_130", "r_same130", "r_neg130", "mono170", "ch3_170",
               "music600"]


@pytest.mark.parametrize("name", MUSIC_CASES)
def test_music_cases_vs_reference(name):
    """add against the oracle (RMS < 1e-5, at most 1 LSB apart on the 16 bit grid), then get on the reference's output: the whole
    document, every sync position identical (none one fine step off), and the same document from the 16 bit entry point"""
    g = G[name]
    x = T.signal(g["signal"])
    assert sha16(O.quantize_sndfile16(x)) == g["input_sha256"]
    H.set_params()
    y = H.add(x, PAYLOAD)
    ref = O.embed(x, O.Key(), PAYLOAD, O.Params()).samples
    assert T.rms(y - ref) < 1e-5, T.rms(y - ref)
    y16, ref16 = O.quantize_sndfile16(y), O.quantize_sndfile16(ref)
    assert np.abs(y16.astype(np.int32) - ref16).max() <= 1
    assert sha16(ref16) == g["output_sha256"]
    doc, trace = get_with_trace(O.int16_to_float(ref16))
    n_real = compare_docs(doc, g["json"])
    assert n_real >= 1 and any(m["bits"] == PAYLOAD for m in doc["matches"])
    n_scores = sum(len(s["scores"]) for s in g["sync"])
    assert compare_sync(trace, g["sync"]) == (n_scores, 0)
    assert H.get_s16(ref16) == doc


def test_music600_two_keys_vs_reference():
    """the 10 min music-like input watermarked once with each of two named keys; get with both keys"""
    g = G["music600_two_keys"]
    ka = O.Key(bytes.fromhex(g["keys"]["alpha"]), "alpha")
    kb = O.Key(bytes.fromhex(g["keys"]["beta"]), "beta")
    x = T.signal(g["signal"])
    y1 = O.int16_to_float(O.quantize_sndfile16(O.embed(x, ka, g["payload"], O.Params()).samples))
    y16 = O.quantize_sndfile16(O.embed(y1, kb, g["payload2"], O.Params()).samples)
    assert sha16(y16) == g["output_sha256"]
    H.set_params()
    doc = H.get(O.int16_to_float(y16), [ka.aes_key, kb.aes_key], ["alpha", "beta"])
    assert compare_docs(doc, g["json"]) >= 2
    assert {(m["key"], m["bits"]) for m in doc["matches"] if m["quality"] > 0.35} >= {("alpha", g["payload"]), ("beta", g["payload2"])}
