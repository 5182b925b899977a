"""Records what the tests compare with the reference project, so that they run without it:

  tests/golden/reference_shader_outputs.npz.xz  the reference's pass shaders (oracle/_ref/shaders): the tests that compare with them
                                                are run with the shaders themselves and tests/oracle_runner.py records, per dispatch,
                                                what it needs to reproduce their outputs (see REFERENCE_GOLDEN there)
  tests/golden/reference_scheduler.json.xz      the reference's host library (oracle/_ref/libnrd_ref.so): its answers to the calls of
                                                tests/test_reference_scheduler.py
  tests/golden/frontend_probe_reference.npz     tests/frontend_probe.cpp compiled against the reference's NRD.hlsli
                                                (oracle/_ref/shaders/frontend_probe_ref): its 400 x 50 table

    python tests/golden/make_reference_golden.py          (from the repository root, after build() where the reference sources are present)

Record again after a change to the scene, the scheduler's calls or the oracle that changes what a recorded test feeds the reference."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)

import oracle_runner as orr  # noqa: E402

SHADER_TESTS = ["tests/test_reference_shaders.py", "tests/test_parity_harness.py::test_reference_shader_mode_of_the_harness"]
SCHEDULER_TESTS = ["tests/test_reference_scheduler.py"]
PROBE = os.path.join(ROOT, "oracle", "_ref", "shaders", "frontend_probe_ref")
PROBE_GOLDEN = os.path.join(ROOT, "tests", "golden", "frontend_probe_reference.npz")


def record_probe():
    """Column 5 is a packed R10G10B10A2 word (uint32); the other columns are float32 values printed with %.9g (exact)."""
    out = subprocess.run([PROBE], check=True, capture_output=True, text=True).stdout
    table = np.array([[float(v) for v in line.split()] for line in out.strip().split("\n")], dtype=np.float64)
    np.savez_compressed(PROBE_GOLDEN, values=np.delete(table, 5, axis=1).astype(np.float32), bits=table[:, 5].astype(np.uint32))


if __name__ == "__main__":
    if not os.path.isdir(os.path.dirname(orr.reference_shader_path("x"))):
        sys.exit("oracle/_ref is not built: build() compiles it where the reference sources are present")
    os.chdir(ROOT)
    record_probe()
    os.environ[orr.RECORD_ENV] = "1"
    os.environ["NRD_B200_RECORD_REFERENCE_SCHEDULER"] = "1"
    r = pytest.main(["-q", "-p", "no:cacheprovider"] + SCHEDULER_TESTS + SHADER_TESTS)
    if r != 0:
        sys.exit("the recorded tests failed (%d); nothing written" % r)
    sys.modules["test_reference_scheduler"].save_recording()
    orr.save_reference_recording()
    for path in (orr.REFERENCE_GOLDEN, sys.modules["test_reference_scheduler"].GOLDEN, PROBE_GOLDEN):
        print("%s: %d bytes" % (path, os.path.getsize(path)))
