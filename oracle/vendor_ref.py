#!/usr/bin/env python
"""Vendor the UNMODIFIED reference package next to the oracle, as part of the build.

    python oracle/vendor_ref.py           # $B200BO_REFERENCE/bayes_opt -> oracle/_ref/bayes_opt

`oracle/_ref/` is git-ignored (never part of the history), exactly like the built `libb200bo.so`: it is a
build product that stays with the built tree, so a machine that runs the tree does not need the reference
source.  The parity tests and the reference arm of bench.py drive the reference's own
`bayes_opt.BayesianOptimization` from it.  Nothing is edited: the
package directory is copied byte for byte by this committed recipe.  Two things the reference needs at
import time and that the image lacks are supplied beside it (they are not reference code):

  * `colorama` (imported by bayes_opt/target_space.py:10 and logger.py:8; not installed, no network)
    -> the stub from oracle/shims/colorama
  * package metadata: bayes_opt/__init__.py:14 asks importlib.metadata for the version of the
    distribution "bayesian-optimization" -> a minimal `*.dist-info/METADATA` with the version of
    /root/reference/pyproject.toml, so that putting oracle/_ref on sys.path is all a caller does.

Product code (bayesianoptimization_b200/) never reads oracle/_ref: it imports `bayes_opt` from wherever
the user's environment provides it; tests/conftest.py and bench.py put oracle/_ref on sys.path (`ref_dir()`,
which only reads: running the tests or the benchmark never copies anything).
"""
from __future__ import annotations

import os
import re
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("B200BO_REFERENCE", "/root/reference")
DST = os.path.join(ROOT, "oracle", "_ref")
# the reference's test modules that exercise the hot path and its callers (SURVEY.md 8a/8c)
REF_TESTS = ("test_acquisition.py", "test_constraint.py", "test_bayesian_optimization.py", "test_target_space.py",
             "test_seq_domain_red.py", "test_parameter.py", "test_util.py", "test_logger.py")


def reference_version() -> str:
    txt = open(os.path.join(REF, "pyproject.toml")).read()
    m = re.search(r'^version\s*=\s*"([^"]+)"', txt, re.M)
    return m.group(1) if m else "0"


def _make_writable(path: str) -> None:
    for base, dirs, files in os.walk(path):
        for n in dirs + files:
            q = os.path.join(base, n)
            os.chmod(q, os.stat(q).st_mode | 0o200)
    os.chmod(path, os.stat(path).st_mode | 0o200)


def ref_dir() -> str | None:
    """The vendored directory to put on sys.path, or None when no build has vendored the reference."""
    return DST if os.path.isdir(os.path.join(DST, "bayes_opt")) else None


def vendor(force: bool = False) -> str | None:
    """Returns the vendored path, or None when the reference tree is not present and nothing was vendored."""
    src = os.path.join(REF, "bayes_opt")
    if not os.path.isdir(src):
        return ref_dir()
    stamp = os.path.join(DST, ".vendored")
    ver = reference_version()
    if (not force and os.path.exists(stamp) and open(stamp).read().strip() == ver
            and all(os.path.exists(os.path.join(DST, "ref_tests", t)) for t in REF_TESTS)):
        return DST
    if os.path.isdir(DST):
        _make_writable(DST)
        shutil.rmtree(DST)
    os.makedirs(DST)
    shutil.copytree(src, os.path.join(DST, "bayes_opt"), ignore=shutil.ignore_patterns("__pycache__"))
    shutil.copytree(os.path.join(ROOT, "oracle", "shims", "colorama"), os.path.join(DST, "colorama"),
                    ignore=shutil.ignore_patterns("__pycache__"))
    _make_writable(DST)  # /root/reference is read-only and copytree keeps the modes
    # the reference's own tests for the path: run on the GPU box against the drop-in (tests/test_gpu_reference_suite.py)
    tdst = os.path.join(DST, "ref_tests")
    os.makedirs(tdst)
    for name in REF_TESTS:
        shutil.copy(os.path.join(REF, "tests", name), os.path.join(tdst, name))
    _make_writable(DST)
    info = os.path.join(DST, f"bayesian_optimization-{ver}.dist-info")
    os.makedirs(info)
    with open(os.path.join(info, "METADATA"), "w") as f:
        f.write(f"Metadata-Version: 2.1\nName: bayesian-optimization\nVersion: {ver}\n")
    with open(os.path.join(info, "RECORD"), "w") as f:
        f.write("")
    with open(stamp, "w") as f:
        f.write(ver + "\n")
    return DST


if __name__ == "__main__":
    p = vendor(force="--force" in sys.argv)
    print(p if p else "reference tree not present; nothing vendored")
