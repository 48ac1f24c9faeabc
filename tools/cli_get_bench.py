"""Wall time and peak RSS of `audiowmark cmp` on a 60 min stereo WAV in tmpfs, at 16 and at 24 bit, for two builds run alternately.

    python tools/cli_get_bench.py --build new=audiowmark_b200 --build parent=<dir with bin/audiowmark> [--minutes 60] [--rounds 3]

The input is seeded noise marked by hostapi.add (so `cmp` finds its payload), written once per bit depth.  Each round runs every
build once per bit depth, builds in turn, so that drift of the machine hits them alike.  Prints one JSON document (also written to
--out): the card name and power limit as nvidia-smi reports them in the same run, and per build and bit depth every wall time and
peak RSS (os.wait4), with their minimum and median."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
PAYLOAD = "f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0f0"


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
        return out.strip().splitlines()[0]
    except (OSError, IndexError):
        return "unknown"


def run(args):
    """-> (seconds, peak RSS in MB, exit code)"""
    t = time.perf_counter()
    p = subprocess.Popen(args, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    _, status, ru = os.wait4(p.pid, 0)
    return time.perf_counter() - t, ru.ru_maxrss / 1024.0, os.waitstatus_to_exitcode(status)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--build", action="append", required=True, help="name=directory that holds bin/audiowmark")
    ap.add_argument("--minutes", type=float, default=60)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    builds = [b.split("=", 1) for b in a.build]
    import awm_testlib as T
    import test_gpu_stream_get as S
    from audiowmark_b200 import hostapi as H
    H.set_params()
    y = H.add(T.noise(a.minutes * 60, 2, seed=60, amp=0.3), PAYLOAD)
    res = {"gpu": gpu_info(), "minutes": a.minutes, "rounds": a.rounds, "what": "audiowmark cmp <file> <payload>, stereo WAV in tmpfs, "
           "wall time incl. process start, CUDA context creation and file I/O", "runs": {}}
    need = 2 * a.minutes * 60 * 44100 * 2 * 5                  # the 16 and the 24 bit file, with room to spare
    tmpfs = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > need else None
    res["dir"] = tmpfs or tempfile.gettempdir()
    with tempfile.TemporaryDirectory(dir=tmpfs) as tmp:
        files = {}
        for bits in (16, 24):
            files[bits] = os.path.join(tmp, "in%d.wav" % bits)
            with open(files[bits], "wb") as f:
                f.write(S.wav_file(S.encode(y, bits, False), 2, bits, False))
        del y
        for r in range(a.rounds):
            for bits in (16, 24):
                for name, d in builds:
                    sec, rss, rc = run([os.path.join(d, "bin", "audiowmark"), "cmp", files[bits], PAYLOAD])
                    res["runs"].setdefault("%s/s%d" % (name, bits), []).append({"s": round(sec, 3), "rss_mb": round(rss, 1), "rc": rc})
    for k, v in res["runs"].items():
        s = sorted(x["s"] for x in v)
        m = sorted(x["rss_mb"] for x in v)
        res.setdefault("summary", {})[k] = {"s_min": s[0], "s_median": s[len(s) // 2], "rss_mb_max": m[-1]}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        open(a.out, "w").write(text + "\n")


if __name__ == "__main__":
    main()
