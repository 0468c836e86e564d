"""The C++ facade (include/neo_b200.hpp) against the reference's own plan/convolver tests restated in tests/cpp/facade_test.cpp."""
import os
import subprocess

import pytest

from conftest import ROOT

BIN = os.path.join(ROOT, "tests", "cpp", "facade_test")


def test_facade_builds_and_reference_dropin_compiles():
    # compile-only everywhere; the drop-in check against the real reference headers is test_reference_dropin_compiles
    proc = subprocess.run(["make", "-C", os.path.join(ROOT, "tests", "cpp")], capture_output=True, text=True)
    assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-2000:]
    assert os.path.exists(BIN)


def test_reference_dropin_compiles():
    # tests/cpp/reference_dropin_check.cpp against the unmodified reference headers (REF in tests/cpp/Makefile), which the repository
    # does not hold: compile-only, and skipped where they are absent
    proc = subprocess.run(["make", "-C", os.path.join(ROOT, "tests", "cpp"), "dropin"], capture_output=True, text=True)
    assert proc.returncode == 0, proc.stdout[-2000:] + proc.stderr[-2000:]
    if "dropin check: ok" not in proc.stdout:
        pytest.skip("the reference headers are not present (REF in tests/cpp/Makefile)")


@pytest.mark.gpu
def test_facade_on_gpu(gpu):
    if not os.path.exists(BIN):
        subprocess.run(["make", "-C", os.path.join(ROOT, "tests", "cpp")], check=True)
    proc = subprocess.run([BIN], capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-2000:]
    assert "all passed" in proc.stdout
