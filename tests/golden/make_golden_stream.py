"""Generate tests/golden/stream_ref.json: what the UNMODIFIED reference (oracle/_ref/audiowmark, built by oracle/Makefile.ref) prints
for `get` and `cmp` on one marked signal stored in every WAV sample format: 8 bit unsigned, 16 / 24 / 32 bit PCM, float32, float64,
RF64 (24 bit) and WAVE_FORMAT_EXTENSIBLE (24 bit).

The signal is a seeded 130 s music signal (tests/awm_testlib.py) marked by the oracle's add on the CPU; the files are built by
tests/test_gpu_stream_get.py (stream_files), which rebuilds them on the GPU box and checks them against the SHA-256 stored here.
Whatever the reference prints is the expected answer; where its WAV reader refuses a format, the refusal (exit code, stderr) is.

Run here (needs /root/reference to build the binary; about a minute):   python tests/golden/make_golden_stream.py
"""
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import build_oracle                 # noqa: E402
import test_gpu_stream_get as S     # noqa: E402

REF = build_oracle.build_reference()
assert REF and os.path.exists(REF), "reference binary not available"


def main():
    files = S.stream_files(S.marked_signal())
    G = {"reference": "swesterfeld/audiowmark 0.6.5 sources compiled unmodified by oracle/Makefile.ref",
         "signal": S.STREAM_SIGNAL, "payload": S.PAYLOAD, "cases": {}}
    with tempfile.TemporaryDirectory(dir="/dev/shm" if os.path.isdir("/dev/shm") else None) as tmp:
        for name, data in files.items():
            path = os.path.join(tmp, name + ".wav")
            open(path, "wb").write(data)
            bits, is_float, container = S.STREAM_CASES[name]
            case = {"bits": bits, "is_float": is_float, "container": container, "sha256": S.sha(data)}
            for cmd, extra in (("get", []), ("cmp", [S.PAYLOAD])):
                p = subprocess.run([REF, cmd, path] + extra, capture_output=True, text=True)
                case[cmd] = {"returncode": p.returncode, "stdout": p.stdout, "stderr": p.stderr.replace(tmp + "/", "")}
                print("%-9s %s rc %d, %d lines" % (name, cmd, p.returncode, len(p.stdout.splitlines())), flush=True)
            G["cases"][name] = case
    out = os.path.join(os.path.dirname(os.path.abspath(__file__)), "stream_ref.json")
    with open(out, "w") as f:
        json.dump(G, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", out)


if __name__ == "__main__":
    main()
