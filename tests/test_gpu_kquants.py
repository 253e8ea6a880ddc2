"""K-quant weights (Q2_K .. Q6_K, SURVEY.md 8f-4) through the C ABI, BIT-EXACT against the reference's own compiled k_quants.c:
quantize_row_q8_K, ggml_vec_dot_q{2..6}_K_q8_K behind ggml_compute_forward_mul_mat, and the same node through the ggml_cuda_* seam.
The weights are seeded random super-blocks (oracle/synth.make_kquant_blocks); what the reference returned for them is recorded in
tests/golden/reference_outputs.json."""
import numpy as np
import pytest

from oracle import bindings as B
from oracle import synth

pytestmark = pytest.mark.gpu

# Q4_K / Q5_K / Q6_K ran bit-exact on a B200 (profiles/r02n_kquant_tests.log).  Q2_K / Q3_K were added after the round's GPU budget was spent: their layout and
# operation order are pinned on the CPU (tests/test_oracle_kquants.py: the numpy restatement the kernel was written from; tests/test_kquants_lane_arithmetic.py: the
# kernel's own word-level index / mask / dp4a / shuffle expressions restated in Python), the CUDA code itself has not met
# hardware yet -- non-strict xfail keeps a first-run surprise from stopping the suite under `-x`; an XPASS is the expected outcome.
_UNRUN = pytest.mark.xfail(strict=False, reason="Q2_K / Q3_K kernels not yet run on a GPU (round-2 GPU budget exhausted); CPU restatement pinned")
KTYPES = [pytest.param(n, t, marks=_UNRUN) if n in ("q2_K", "q3_K") else (n, t) for n, t in B.KQUANT_TYPES.items()]


@pytest.fixture(scope="module")
def L():
    from llm_b200 import _lib
    lib = _lib.lib()
    assert lib.b200_init(0) == 0
    return lib


@pytest.fixture(scope="module")
def ctx():
    from llm_b200 import ggml
    c = ggml.Context()
    yield c
    c.close()


def acts(rng, Bn, K):
    x = (rng.standard_normal((Bn, K)) * rng.uniform(0.05, 8, (Bn, 1))).astype(np.float32)
    if Bn > 2:
        x[1, :256] = 0.0                                   # an all-zero super-block: d = 0, quants 0
        x[2] = np.round(x[2] * 4) / 4                      # many ties in |x| and exact .5 products
        x[2, 5] = -x[2].max(); x[2, 9] = x[2].max()        # equal magnitudes, opposite signs: the FIRST one sets the scale's sign
    return x


def q8_K_inputs():
    return acts(np.random.default_rng(11), 9, 4096)


def test_quantize_q8_K_bit_exact(L, reference):
    x = q8_K_inputs()
    Bn, K = x.shape
    got = np.empty((Bn, K // 256, 292), np.uint8)
    assert L.b200_op_quantize_q8_K(x.ctypes.data, K, Bn, got.ctypes.data) == 0
    zero = got[:, :, :4].copy().view(np.float32)[:, :, 0] == 0.0             # the reference leaves bsums of an all-zero super-block unwritten:
    got[zero, 260:] = 0                                                     # they are recorded as zeros
    reference("kquant/quantize_q8_K", got)


MUL_MAT_SHAPES = [(4096, 130, 1), (11008 // 256 * 256, 64, 1), (256, 33, 5), (5120, 96, 7), (1024, 257, 33)]


def mul_mat_inputs(t, K, N, Bn):
    seed = K * 3 + N + t
    return synth.make_kquant_blocks(t, N, K, seed), acts(np.random.default_rng(seed), Bn, K)


@pytest.mark.parametrize("name,t", KTYPES)
@pytest.mark.parametrize("K,N,Bn", MUL_MAT_SHAPES)
def test_mul_mat_kquant_bit_exact(L, reference, name, t, K, N, Bn):
    wq, x = mul_mat_inputs(t, K, N, Bn)
    got = np.empty((Bn, N), np.float32)
    assert L.b200_op_mul_mat(t, wq.ctypes.data, K, N, x.ctypes.data, Bn, got.ctypes.data, 0) == 0
    reference(f"kquant/mul_mat/{name}/K{K} N{N} B{Bn}", got)


def seam_inputs(t):
    """-> weights [96, 1024] and the activations of batches 1, 4 and 33"""
    rng = np.random.default_rng(17 + t)
    K, N = 1024, 96
    return synth.make_kquant_blocks(t, N, K, 17 + t), [rng.standard_normal((Bn, K)).astype(np.float32) for Bn in (1, 4, 33)]


@pytest.mark.parametrize("name,t", KTYPES)
def test_seam_mul_mat_kquant(ctx, reference, name, t):
    """the node the reference executor sends: src0 uploaded with ggml_cuda_transform_tensor (GGML super-blocks as they are), src1 / dst on the host"""
    wq, xs = seam_inputs(t)
    N, K = wq.shape[0], xs[0].shape[1]
    for x in xs:
        w = ctx.transfer_to_gpu(ctx.quantized(t, wq, K))
        dst = ctx.op_mul_mat(w, ctx.from_numpy(x))
        assert ctx.compute(dst, nth=4) is True
        got = ctx.host_array(dst).reshape(x.shape[0], N)
        reference(f"kquant/seam/{name}/B{x.shape[0]}", got)


def test_kquant_rejects_bad_shapes(L):
    x = np.zeros((1, 128), np.float32); w = np.zeros(144, np.uint8); o = np.zeros((1, 1), np.float32)
    assert L.b200_op_mul_mat(B.Q4_K, w.ctypes.data, 128, 1, x.ctypes.data, 1, o.ctypes.data, 0) != 0        # K % 256
    x = np.zeros((1, 256), np.float32)
    assert L.b200_op_mul_mat(B.Q4_K, w.ctypes.data, 256, 1, x.ctypes.data, 1, o.ctypes.data, 7) != 0        # no tensor-core variant for K-quants
