"""Generate tests/golden/cli_ref.json with the UNMODIFIED reference built by oracle/Makefile.ref (oracle/_ref/audiowmark):
exit code, stdout, stderr and output file SHA-256 of every command tests/test_cli_vs_ref_cpu.py runs, in the same order and
in the same kind of scratch directory.

Run where the reference sources can be built:   python tests/golden/make_golden_cli.py
"""
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")]
import build_oracle                 # noqa: E402
import test_cli_vs_ref_cpu as C     # noqa: E402

REF = build_oracle.build_reference()
assert REF and os.path.exists(REF), "reference binary not available"


def main():
    G = {"helper_sequence": [], "argv_cases": []}
    with tempfile.TemporaryDirectory() as tmp:
        for args, out in C.HELPER_SEQUENCE:
            r = C.run(REF, tmp, args)
            G["helper_sequence"].append(dict(args=args, **r, sha256=C.digest(os.path.join(tmp, out)) if out else None))
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.check_call([REF] + C.ARGV_SETUP, cwd=tmp)
        for args in C.ARGV_CASES:
            G["argv_cases"].append(dict(args=args, **C.run(REF, tmp, args)))
    with open(C.GOLDEN, "w") as f:
        json.dump(G, f, indent=1)
        f.write("\n")
    print("wrote", C.GOLDEN)


if __name__ == "__main__":
    main()
