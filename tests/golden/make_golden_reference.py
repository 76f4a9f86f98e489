"""Record into tests/golden/reference/ what the reference's own lines (oracle/_ref) return to every helper wrapped by
util.recorded, so that the comparisons with the reference run where it cannot be built.  Run where oracle/_ref is built
(`make -C oracle ref` with the reference sources at REF):

    python tests/golden/make_golden_reference.py

It runs the CPU tests that call the reference with recording on, then the reference calls of the GPU tests' fixtures.
Recordings are keyed by the helper's arguments: rerun it after changing what a test passes to the reference."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, TESTS)
os.environ["B200_RECORD_REFERENCE"] = "1"

import util  # noqa: E402

assert util.ref("strict") is not None and util.ref("fast") is not None, "build oracle/_ref first (make -C oracle ref)"
subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider", "-m", "not gpu"]
               + [os.path.join(TESTS, f) for f in sorted(os.listdir(TESTS)) if f.startswith("test_cpu_")], check=True, cwd=os.path.dirname(TESTS))

import test_filmic_gpu as tf  # noqa: E402

for name in tf.CASES:
    tf.data_blob(name)
tf.legacy_live_blobs()
