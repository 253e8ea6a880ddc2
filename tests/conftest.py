import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

# the oracle's OpenMP loops are tiny; 128 threads per process under pytest-xdist oversubscribes the GPU box's host badly
os.environ.setdefault("OMP_NUM_THREADS", "8")
os.environ.setdefault("OMP_WAIT_POLICY", "passive")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "slow: takes more than a few seconds")


def _ensure_oracle():
    """tests may build the checker (oracle/liboracle.so is plain C, no reference sources needed)."""
    so = os.path.join(ROOT, "oracle", "liboracle.so")
    if not os.path.exists(so):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "liboracle.so"])
    return so


@pytest.fixture(scope="session")
def orc():
    _ensure_oracle()
    from oracle import bindings as B
    return B.Oracle()


@pytest.fixture(scope="session")
def ref():
    """The reference's own compiled ggml.c (oracle/_ref), which build() makes only where the reference's sources are at hand."""
    from oracle import bindings as B
    if not B.have_ref("ref"):
        pytest.skip("oracle/_ref/libggml_ref.so not built (needs the reference's sources)")
    return B.RefLib("ref")


def fingerprint(a):
    """How tests/golden/reference_outputs.json records an output of the reference: dtype, size and the SHA-256 of the bytes."""
    a = np.ascontiguousarray(a)
    return {"dtype": str(a.dtype), "size": int(a.size), "sha256": hashlib.sha256(a.tobytes()).hexdigest()}


@pytest.fixture(scope="session")
def reference():
    """reference(key, got) asserts that `got` is, bit for bit, what the reference's compiled ggml.c returned for the same seeded inputs
    (recorded by oracle/gen_reference_outputs.py)."""
    table = json.load(open(os.path.join(GOLDEN, "reference_outputs.json")))

    def check(key, got):
        want, mine = table[key], fingerprint(got)
        assert mine == want, f"{key}: not bit-identical to the reference ({mine['dtype']}[{mine['size']}] vs {want['dtype']}[{want['size']}])"
    return check


@pytest.fixture(scope="session")
def golden_ops():
    return np.load(os.path.join(GOLDEN, "ops.npz"))


def has_gpu():
    try:
        import ctypes
        cudart = ctypes.CDLL("libcudart.so")
        n = ctypes.c_int(0)
        return cudart.cudaGetDeviceCount(ctypes.byref(n)) == 0 and n.value > 0
    except OSError:
        try:
            import torch
            return torch.cuda.is_available()
        except Exception:
            return False
