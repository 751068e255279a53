#!/usr/bin/env python3
"""Regenerates tests/golden/ref_digests.json.

Runs the tests that compare the oracle or the GPU with the reference's own functions (test_oracle_vs_ref.py,
test_cpu_ref_replay.py, test_gpu_dsp_table.py) with REF_DIGESTS_OUT set: each test case compares every output with the
live reference and then stores the SHA-256 of those outputs under its test id (oracle_lib.RefDigest).  Without the
reference the same tests compare with these digests.  Needs oracle/_ref built from the reference sources
(`make -C oracle ref`) and, for test_gpu_dsp_table.py, a B200; extra arguments go to pytest (e.g. -m "not gpu").
REF_DIGESTS_OUT=<file> writes somewhere else; digests already in the file are kept unless a test replaces them.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
MODULES = ["tests/test_oracle_vs_ref.py", "tests/test_cpu_ref_replay.py", "tests/test_gpu_dsp_table.py"]


def main():
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_shim.so")):
        sys.exit("oracle/_ref is not built: the digests must come from the live reference")
    env = dict(os.environ, REF_DIGESTS_OUT=os.environ.get("REF_DIGESTS_OUT", os.path.join(HERE, "ref_digests.json")))
    sys.exit(subprocess.call([sys.executable, "-m", "pytest", "-q", *MODULES, *sys.argv[1:]], cwd=ROOT, env=env))


if __name__ == "__main__":
    main()
