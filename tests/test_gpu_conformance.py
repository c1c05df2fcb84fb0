"""SURVEY.md 8(f) rank 1: the reference's test matrix (src/test.cpp:76-179: 10 key types x 14 payload shapes
x separate/combined x ascending/descending x 8 distributions, sizes 1..10^4) run against the GPU path through the
C ABI by tests/cpp/conformance_b200.cpp, with its own generators and a check stricter than the reference's
checkData().

The driver is built by `make -C oracle conformance`, part of __graft_entry__.build()."""
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
EXE = ROOT / "oracle" / "_build" / "conformance_b200"


def _ensure_built():
    if not EXE.exists():
        subprocess.run(["make", "-C", str(ROOT / "oracle"), "conformance"], check=True, capture_output=True)
    return EXE.exists()


def test_conformance_driver_fails_loudly_without_gpu():
    """CPU box: the driver links against libb200sort.so and must stop at the first sort (no fallback)"""
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("no-GPU behaviour")
    except ImportError:
        pass
    assert _ensure_built()
    r = subprocess.run([str(EXE), "10", "42"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 3 and "no CPU fallback" in r.stdout, r.stdout[-500:]


@pytest.mark.gpu
def test_reference_test_matrix_passes_on_the_gpu_path():
    assert _ensure_built(), "oracle/_build/conformance_b200 missing: run __graft_entry__.build()"
    r = subprocess.run([str(EXE), "10000", "42"], capture_output=True, text=True, timeout=1500)
    tail = r.stdout[-1500:]
    assert r.returncode == 0 and "All tests passed" in r.stdout, tail
    assert "FAILED" not in r.stdout
    # 5 sizes x 4 (separate/combined x up/down) x 10 key types x 14 payload shapes x 8 distributions, minus the
    # combined records whose size is not a power of two
    n_tests = r.stdout.count("passed\n") - 1
    assert n_tests > 10000, n_tests
