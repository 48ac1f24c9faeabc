"""CPU: the host-only commands and the argv handling of bin/audiowmark against the reference binary built by oracle/Makefile.ref.
The reference's answers -- exit code, stdout, stderr and the SHA-256 of every output file -- are stored in
tests/golden/cli_ref.json (made by tests/golden/make_golden_cli.py from the command lists below); bin/audiowmark has to give
the same answers, byte for byte."""
import hashlib
import json
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "audiowmark_b200", "bin", "audiowmark")
GOLDEN = os.path.join(ROOT, "tests", "golden", "cli_ref.json")

# run in this order in one directory: (argv, output file to compare or None)
HELPER_SEQUENCE = [
    (["test-gen-noise", "n16.wav", "3", "44100"], "n16.wav"),
    (["test-gen-noise", "--bits", "24", "n24.wav", "2", "48000"], "n24.wav"),
    (["test-gen-noise", "--bits", "32", "n32.wav", "1.5", "22050"], "n32.wav"),
    (["test-gen-noise", "--test-key", "5", "nk.wav", "1", "8000"], "nk.wav"),
    (["cut-start", "n16.wav", "c.wav", "1000"], "c.wav"),
    (["test-info", "n16.wav", "frames"], None), (["test-info", "n24.wav", "bit_depth"], None),
    (["test-info", "n32.wav", "sample_rate"], None), (["test-info", "n16.wav", "channels"], None),
    (["test-subtract", "n16.wav", "n16.wav", "z.wav"], "z.wav"),
    (["test-snr", "n16.wav", "n16.wav"], None),
    (["gentest", "n16.wav", "g.wav"], None),                      # input too short: same complaint, no file
    (["test-clip", "n16.wav", "clip.wav", "3", "1"], "clip.wav"),
    (["test-clip", "--test-key", "2", "n16.wav", "clip2.wav", "7", "2"], "clip2.wav"),
    (["test-speed", "--test-key", "3", "5"], None),
]

# run in this order in one directory that holds ARGV_SETUP's n.wav
ARGV_SETUP = ["test-gen-noise", "n.wav", "1", "44100"]
ARGV_CASES = [
    [], ["foo"], ["--foo"], ["add"], ["add", "a.wav"], ["add", "a.wav", "b.wav"], ["get"], ["cmp", "x.wav"],
    ["add", "--strength", "abc", "a.wav", "b.wav", "00"], ["add", "--short", "13", "a.wav", "b.wav", "abc"], ["add", "--bogus", "a.wav", "b.wav", "00"],
    ["get", "--bogus", "a.wav"], ["get", "--strength", "10", "a.wav"], ["get", "--n-best", "-1", "n.wav"],
    ["get", "--detect-speed", "--detect-speed-patient", "n.wav"], ["gen-key"], ["gen-key", "k1", "k2"], ["test-info", "n.wav", "bogus"],
    ["test-gen-noise", "x.wav", "abc", "44100"], ["cut-start", "n.wav"], ["test-change-speed", "n.wav", "o.wav"],
    ["add", "--key", "nokey.key", "n.wav", "o.wav", "00"], ["add", "--test-key", "1", "--key", "x", "n.wav", "o.wav", "00"],
    ["add", "--format", "bogus", "n.wav", "o.wav", "00"], ["add", "--raw-rate", "x", "n.wav", "o.wav", "00"],
    ["add", "n.wav", "o.wav", "xyz"], ["add", "nofile.wav", "o.wav", "00"], ["get", "nofile.wav"], ["cmp", "nofile.wav", "00"],
    ["get", "--try-speed", "abc", "n.wav"], ["get", "--json"],
    # the generic option scanner against the reference's hand-written sequences: repeated flags, "=" forms, last value wins,
    # "--a || --b" pairs, options after positional arguments, checks that fire before later conversions
    ["get", "--hard", "--hard", "n.wav"], ["get", "--n-best=-1", "n.wav"], ["add", "--format", "raw", "--format", "bogus", "a", "b", "00"],
    ["add", "--strength"], ["-q", "foo"], ["--strict"], ["add", "a.wav", "--bogus", "b.wav", "00"],
    ["get", "--input-format", "raw", "--format", "bogus", "n.wav"], ["get", "--raw-bits", "16", "n.wav"],
    ["add", "--input-format", "rf64", "--strength", "abc", "n.wav", "o.wav", "00"], ["get", "--chunk-size", "5", "n.wav"],
    ["cmp", "--expect-matches", "x", "n.wav", "00"], ["test-gen-noise", "--bits", "x", "o.wav", "1", "44100"],
    ["get", "--detect-speed", "--try-speed", "1.1", "--test-speed", "abc", "n.wav"], ["add", "--raw-encoding", "double", "--raw-bits", "16", "n.wav", "o.wav", "00"], ["add", "--raw-rate", "0x", "n.wav", "o.wav", "00"],
    ["add", "--raw-encoding", "float", "--raw-bits", "12", "--raw-endian", "middle", "n.wav", "o.wav", "00"],
    ["add", "--short", "12", "n.wav", "o.wav", "abcd"], ["add", "--short=16", "--short", "13", "n.wav", "o.wav", "abcd"],
    ["test-clip", "--test-key", "1", "--test-key", "2", "n.wav", "c.wav", "1", "1"], ["get", "--key"], ["get", "--key=nokey.key", "n.wav"],
    ["cut-start", "n.wav", "o.wav", "abc"], ["test-speed", "x"],
]


def run(binary, cwd, args):
    p = subprocess.run([binary] + args, capture_output=True, text=True, cwd=cwd)
    return {"rc": p.returncode, "stdout": p.stdout, "stderr": p.stderr}


def digest(path):
    return hashlib.sha256(open(path, "rb").read()).hexdigest() if os.path.exists(path) else None


def golden():
    return json.load(open(GOLDEN))


def test_helper_commands_write_identical_files(tmp_path):
    want = golden()["helper_sequence"]
    assert [w["args"] for w in want] == [args for args, _ in HELPER_SEQUENCE]
    for (args, out), w in zip(HELPER_SEQUENCE, want):
        assert run(CLI, tmp_path, args) == {k: w[k] for k in ("rc", "stdout", "stderr")}, args
        if out:
            assert w["sha256"] is not None and digest(tmp_path / out) == w["sha256"], args


def test_argv_errors_are_the_reference_ones(tmp_path):
    want = golden()["argv_cases"]
    assert [w["args"] for w in want] == ARGV_CASES
    subprocess.check_call([CLI] + ARGV_SETUP, cwd=tmp_path)
    for args, w in zip(ARGV_CASES, want):
        assert run(CLI, tmp_path, args) == {k: w[k] for k in ("rc", "stdout", "stderr")}, args
