"""Generate tests/golden/golden_large.json: BASELINE.json's configs 2-4 at their stated sizes, the digital-silence cases, the
music-like / tonal / quiet / clipped / one-sided stereo / mono / 3-channel cases (MUSIC_CASES) and the exact sync positions, all
from the UNMODIFIED reference sources built by oracle/Makefile.ref
  oracle/_ref/audiowmark   the reference CLI
  oracle/_ref/sync_dump    the reference's SyncFinder::search behind a print loop (oracle/ref_shims/sync_dump.cc)

Run here (needs /root/reference to build the binaries; about 10 minutes):   python tests/golden/make_golden_large.py
Only some of MUSIC_CASES (about 10 s each, music600 2 minutes), the rest of the file kept:   python tests/golden/make_golden_large.py music130 ...
A full run reproduces the MUSIC_CASES entries byte for byte; of the older entries, the hour's add_stderr holds the temporary
directory of the run that made it, and the reference prints the rating of some of the hour's and speed600's patterns with a
last digit that can change from run to run (143.98074 / 143.98073).
Only hashes, JSON documents and score lists are stored; the tests regenerate the inputs from seeds with the oracle
(bit exact against these hashes) on whatever box they run.
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import awm_oracle as O      # noqa: E402
import awm_testlib as T     # noqa: E402
import build_oracle         # noqa: E402

REF = build_oracle.build_reference()
DUMP = build_oracle.REF_SYNC_DUMP
assert REF and os.path.exists(REF) and os.path.exists(DUMP), "reference binaries not available"
PAYLOAD = "f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0"
PAYLOAD2 = "0123456789abcdef0123456789abcdef"
TWO_KEYS = {"alpha": "000102030405060708090a0b0c0d0e0f", "beta": "101112131415161718191a1b1c1d1e1f"}


def _sig(fn, **args):
    return {"fn": fn, "args": args}


# name -> input (tests/awm_testlib.py signal spec); every case is watermarked by the reference with PAYLOAD and read back
MUSIC_CASES = {
    "music130": _sig("music", seconds=130, channels=2, seed=1),
    "tone170": _sig("tone", seconds=170, channels=2, seed=2),
    "quiet130": _sig("quiet", seconds=130, channels=2, seed=3),
    "dc_clip130": _sig("dc_clip", seconds=130, channels=2, seed=4),
    "r_zero130": _sig("one_sided", seconds=130, kind="zero", seed=5),
    "r_m50_130": _sig("one_sided", seconds=130, kind="m50", seed=5),
    "r_same130": _sig("one_sided", seconds=130, kind="same", seed=5),
    "r_neg130": _sig("one_sided", seconds=130, kind="neg", seed=5),
    "mono170": _sig("music", seconds=170, channels=1, seed=6),
    "ch3_170": _sig("music", seconds=170, channels=3, seed=7),
    "music600": _sig("music", seconds=600, channels=2, seed=8),
}


def run(exe, *args, ok_codes=(0,)):
    t = time.time()
    p = subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True)
    assert p.returncode in ok_codes, (args, p.returncode, p.stderr)
    print("  %-60s %.1f s" % (" ".join([os.path.basename(exe)] + [str(a) for a in args])[:60], time.time() - t), flush=True)
    return p


def sha(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def pcm16(path):
    x, rate, bits = O.read_wav(path)
    return O.quantize_sndfile16(x)


def sync_dump(path):
    """-> list of searches: {"mode", "n_frames", "scores": [[index, quality, "A"|"B"], ...]} in call order"""
    out = []
    for line in run(DUMP, path).stdout.splitlines():
        w = line.split()
        if w[0] == "search":
            out.append({"mode": w[1], "n_frames": int(w[2]), "scores": []})
        elif w[0] == "score":
            out[-1]["scores"].append([int(w[1]), float(w[2]), w[3]])
    return out


def get_case(tmp, wav, extra=()):
    js = os.path.join(tmp, "out.json")
    g = run(REF, "get", *extra, "--json", js, wav)
    return {"get_stdout": g.stdout, "json": json.load(open(js)), "get_args": list(extra)}


def music_cases(G, tmp, names):
    """MUSIC_CASES (and music600_two_keys with music600).  130 s: one full A block, and short enough (< 3.1 blocks) that the clip
    decoder's two CLIP searches run too; 170 s: BLOCK search only, three sync blocks.  The temporary directory is cut out of the
    stored add output, so that a second run stores the same bytes."""
    p = lambda name: os.path.join(tmp, name)
    for name in names:
        spec = MUSIC_CASES[name]
        x = T.signal(spec)
        O.write_wav16(p("m.wav"), x)
        a = run(REF, "add", p("m.wav"), p("mwm.wav"), PAYLOAD)
        G[name] = dict(get_case(tmp, p("mwm.wav")), signal=spec, input_sha256=sha(O.quantize_sndfile16(x)), add_stderr=a.stderr.replace(tmp + "/", ""),
                       output_sha256=sha(pcm16(p("mwm.wav"))), payload=PAYLOAD, sync=sync_dump(p("mwm.wav")))
        if name == "music600":
            # the same input watermarked twice with two named keys from key files (as two_keys30 in golden.json); get with both
            k1, k2 = p("k1.key"), p("k2.key")
            open(k1, "w").write('key %s\nname "alpha"\n' % TWO_KEYS["alpha"])
            open(k2, "w").write('key %s\nname "beta"\n' % TWO_KEYS["beta"])
            run(REF, "add", "--key", k1, p("m.wav"), p("k1wm.wav"), PAYLOAD)
            a2 = run(REF, "add", "--key", k2, p("k1wm.wav"), p("k2wm.wav"), PAYLOAD2)
            js = p("out.json")
            g2 = run(REF, "get", "--key", k1, "--key", k2, "--json", js, p("k2wm.wav"))
            G["music600_two_keys"] = {"signal": spec, "keys": TWO_KEYS, "payload": PAYLOAD, "payload2": PAYLOAD2,
                                      "add_stderr": a2.stderr.replace(tmp + "/", ""), "output_sha256": sha(pcm16(p("k2wm.wav"))),
                                      "get_stdout": g2.stdout, "json": json.load(open(js))}


def main():
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden_large.json")
    names = sys.argv[1:]
    assert all(n in MUSIC_CASES for n in names), "unknown case; one of %s" % ", ".join(MUSIC_CASES)
    if names:                                       # only these cases, the rest of the file stays as it is
        G = json.load(open(out))
        with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
            music_cases(G, tmp, names)
        json.dump(G, open(out, "w"), indent=1, sort_keys=True)
        print("wrote", out, os.path.getsize(out), "bytes")
        return
    G = {"reference": "swesterfeld/audiowmark 0.6.5 sources compiled unmodified by oracle/Makefile.ref (FFT: oracle/ref_shims/fftw_shim.cc, "
                      "resampler: oracle/ref_shims/awm_vresampler.hh); sync positions from oracle/ref_shims/sync_dump.cc"}
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        p = lambda name: os.path.join(tmp, name)
        # ---- digital silence: every sync quality is exactly 0, every soft bit 0/0 (VERDICT r1 item 1)
        O.write_wav16(p("z170.wav"), np.zeros((170 * 44100, 2), np.float32))
        G["silence170"] = dict(get_case(tmp, p("z170.wav")), seconds=170, sync=sync_dump(p("z170.wav")))
        # 60 s of watermarked noise followed by 60 s of zeros (short file: clip decoder runs as well)
        x60 = O.int16_to_float(O.quantize_sndfile16(T.noise(60.0, 2, seed=4321)))
        O.write_wav16(p("n60.wav"), x60)
        run(REF, "add", p("n60.wav"), p("n60wm.wav"), PAYLOAD)
        y60 = pcm16(p("n60wm.wav"))
        ns = np.concatenate([y60, np.zeros((60 * 44100, 2), np.int16)])
        O.write_wav16(p("ns.wav"), O.int16_to_float(ns))
        G["noise60_silence60"] = dict(get_case(tmp, p("ns.wav")), noise_seed=4321, wm_sha256=sha(y60), input_sha256=sha(ns), sync=sync_dump(p("ns.wav")))

        # ---- config 2: 1 h stereo reference noise (test-gen-noise), add + get, 3 chunks
        run(REF, "test-gen-noise", p("h.wav"), 3600, 44100)
        a = run(REF, "add", p("h.wav"), p("hwm.wav"), PAYLOAD)
        h16 = pcm16(p("hwm.wav"))
        G["hour"] = dict(get_case(tmp, p("hwm.wav")), input_sha256=sha(pcm16(p("h.wav"))), output_sha256=sha(h16), add_stderr=a.stderr,
                         payload=PAYLOAD, sync=sync_dump(p("hwm.wav")))
        c = run(REF, "cmp", p("hwm.wav"), PAYLOAD, ok_codes=(0, 1))
        G["hour"]["cmp_tail"] = c.stdout.splitlines()[-2:]
        # first 140 s of the output: what the test-clip case below and cheap tests can regenerate without the whole hour
        G["hour"]["output_head140_sha256"] = sha(h16[:140 * 44100])
        G["hour"]["output_head600_sha256"] = sha(h16[:600 * 44100])

        # ---- config 3: 30 s clip cut from the 1 h output by the reference's test-clip (seed 0)
        run(REF, "test-clip", p("hwm.wav"), p("clip.wav"), 0, 30)
        c16 = pcm16(p("clip.wav"))
        # locate the cut (start point is a keyed random position inside the first two blocks, src/audiowmark.cc:362-372)
        first = h16[:2 * 2226 * 1024 + 31 * 44100]
        key = c16[:64].tobytes()
        start = None
        hb = first.tobytes()
        pos = hb.find(key)
        while pos >= 0:
            if pos % 4 == 0 and np.array_equal(first[pos // 4: pos // 4 + len(c16)], c16):
                start = pos // 4
                break
            pos = hb.find(key, pos + 1)
        assert start is not None
        G["clip30"] = dict(get_case(tmp, p("clip.wav")), start_frame=int(start), n_frames=int(len(c16)), input_sha256=sha(c16), sync=sync_dump(p("clip.wav")))

        # ---- config 4: --detect-speed on 10 min stereo, speeds at and inside the +-10 % edges of the scan range.
        # NOTE: everything behind a resampler runs on oracle/ref_shims/awm_vresampler.hh (zita-resampler is absent).
        O.write_wav16(p("m10.wav"), O.int16_to_float(h16[:600 * 44100]))
        G["speed600"] = {"cases": []}
        for speed in (0.9, 0.9764, 1.01, 1.1):
            run(REF, "test-change-speed", p("m10.wav"), p("sp.wav"), speed)
            s16 = pcm16(p("sp.wav"))
            case = get_case(tmp, p("sp.wav"), extra=("--detect-speed",))
            case.update(speed=speed, input_sha256=sha(s16), n_frames=int(len(s16)))
            G["speed600"]["cases"].append(case)
        music_cases(G, tmp, MUSIC_CASES)
    json.dump(G, open(out, "w"), indent=1, sort_keys=True)
    print("wrote", out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
