"""Pins the numpy restatement of the K-quant path (oracle/kquants_np.py) to the reference's own compiled k_quants.c, bit for bit:
quantize_row_q8_K and ggml_vec_dot_q{2..6}_K_q8_K behind ggml_compute_forward_mul_mat.  CPU only; what the reference returned for these
inputs is in tests/golden/kquants_ref.npz (oracle/gen_reference_outputs.py)."""
import os

import numpy as np
import pytest

from oracle import bindings as B
from oracle import kquants_np as KN

from conftest import GOLDEN


def recorded():
    return np.load(os.path.join(GOLDEN, "kquants_ref.npz"))


def _inputs():
    rng = np.random.default_rng(1)
    K = 512
    x = (rng.standard_normal((3, K)) * rng.uniform(0.1, 5, (3, 1))).astype(np.float32)
    x[1, :256] = 0.0
    x[2] = np.round(x[2] * 4) / 4
    x[2, 5] = -np.abs(x[2]).max(); x[2, 9] = np.abs(x[2]).max()          # equal magnitudes, opposite signs: the first sets the scale's sign
    w = (rng.standard_normal((4, K)) / 22).astype(np.float32)
    w[:, :16] *= 8.0
    return K, x, w


def test_quantize_row_q8_K_matches_the_reference():
    K, x, _ = _inputs()
    ref = recorded()
    for b in range(x.shape[0]):
        mine = KN.q8_K_bytes(KN.quantize_row_q8_K(x[b])).reshape(-1, 292)
        want = ref[f"q8_K_row{b}"].reshape(-1, 292)
        zero = want[:, :4].copy().view(np.float32)[:, 0] == 0.0            # bsums of an all-zero super-block are left unwritten by the reference
        assert np.array_equal(mine[:, :260], want[:, :260])
        assert np.array_equal(mine[~zero, 260:], want[~zero, 260:])


@pytest.mark.parametrize("name,t", list(B.KQUANT_TYPES.items()))
def test_vec_dot_kquant_matches_the_reference(name, t):
    K, x, _ = _inputs()
    ref = recorded()
    wq, want = ref[f"{name}_wq"], ref[f"{name}_mul_mat"]           # the reference's quantize_row_{name} of _inputs()'s w, and its mul_mat
    for b in range(x.shape[0]):
        xq = KN.quantize_row_q8_K(x[b])
        for n in range(wq.shape[0]):
            got = KN.vec_dot(t, wq[n], xq)
            assert got.view(np.uint32) == want[b, n].view(np.uint32), (name, b, n, got, want[b, n])
