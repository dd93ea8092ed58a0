"""The reference's own test modules, rebound to the drop-in (tests/ref_suite_plugin.py), on a box without a GPU:
everything that does not touch the device must pass, and every failure must be the engine's loud
"no CUDA device ... no CPU fallback" error - never a silent CPU path, never an API mismatch."""
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SUITE = os.path.join(ROOT, "oracle", "_ref", "ref_tests")


def run_reference_suite(extra=()):
    env = dict(os.environ, PYTHONPATH=os.path.join(ROOT, "tests") + os.pathsep + os.environ.get("PYTHONPATH", ""))
    # --confcutdir: with `-c /dev/null` pytest would otherwise collect every parent directory of the suite up to
    # the filesystem root, and fail on one the user may not list.
    cmd = [sys.executable, "-m", "pytest", "-q", "-p", "ref_suite_plugin", "-p", "no:cacheprovider", "--tb=line",
           "-c", os.devnull, "--rootdir", SUITE, "--confcutdir", SUITE, SUITE, *extra]
    return subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1500)


@pytest.mark.skipif(torch.cuda.is_available(), reason="GPU present: tests/test_gpu_reference_suite.py runs the suite")
def test_reference_suite_without_gpu_fails_only_with_the_loud_device_error():
    if not os.path.isdir(SUITE):
        pytest.skip("reference tests not vendored (build() runs oracle/vendor_ref.py where the reference is present)")
    out = run_reference_suite().stdout
    m = re.search(r"(\d+) failed, (\d+) passed", out)
    assert m, out[-2000:]
    failed, passed = int(m.group(1)), int(m.group(2))
    assert passed >= 100  # constructors, parameter validation, target space, serialisation paths ...
    errors = [ln for ln in out.splitlines() if re.match(r"^(E   |/).*(Error|assert)", ln)]
    other = [ln for ln in errors if "no CUDA device available" not in ln and "pop from an empty deque" not in ln]
    assert not other, "\n".join(other[:20])
    assert failed == sum("no CUDA device available" in ln for ln in errors if ln.startswith("/"))
