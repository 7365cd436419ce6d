"""CPU: the reference's OWN test-suite run against this repo's `real_time_vad` package (286 cases, every model call
mocked at the `ort.InferenceSession` / `VADProcessor` seams).  The reference itself scores 284/286 on it: the two
failures are defects of its tests (test_audio_utils.py:100-110 expects noise subtraction from a gate, :226-236 overflows
int32 under numpy 2) -- SURVEY.md section 4.  A drop-in must score the same.

The suite belongs to the reference project (Picurit/cutter-vad) and is not part of this repository: set
CVAD_REFERENCE_TESTS to the `tests/` directory of a checkout of the reference to run it; without it the test skips."""
import os
import re
import shutil
import subprocess
import sys
from pathlib import Path

import pytest

from conftest import ORACLE, PKG

REF_TESTS = os.environ.get("CVAD_REFERENCE_TESTS", "")


@pytest.mark.skipif(not REF_TESTS, reason="CVAD_REFERENCE_TESTS (the reference checkout's tests/ directory) is not set")
def test_reference_suite_passes_against_this_package(tmp_path):
    assert Path(REF_TESTS).is_dir(), f"CVAD_REFERENCE_TESTS={REF_TESTS} is not a directory"
    work = tmp_path / "reftests"
    shutil.copytree(REF_TESTS, work)
    env = dict(os.environ)
    # oracle/ort_shim only satisfies the suite's own `import onnxruntime`; the package never imports it
    env["PYTHONPATH"] = os.pathsep.join([str(PKG), str(ORACLE / "ort_shim"), str(ORACLE)])
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", str(work)],
                       capture_output=True, text=True, env=env, cwd=str(work), timeout=900)
    tail = r.stdout[-2000:]
    m = re.search(r"(\d+) failed, (\d+) passed", tail)
    assert m, tail
    failed = set(re.findall(r"FAILED \S+::(\w+)", tail))
    assert failed == {"test_denoise_audio", "test_float32_to_pcm_32bit"}, tail
    assert int(m.group(2)) == 284, tail
