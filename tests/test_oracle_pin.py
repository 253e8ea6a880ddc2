"""Pins the oracle: the plain-C restatement against what the reference's own compiled ggml.c returned for the same seeded inputs --
(1) the golden vectors of oracle/gen_golden.py and (2) the recorded outputs of oracle/gen_reference_outputs.py.
Bit-exact everywhere (integer/byte work and f32 with the reference's own operation order)."""
import os

import numpy as np
import pytest

from oracle import bindings as B
from oracle import synth
from oracle.gen_golden import MICRO, synthetic_cos

from conftest import GOLDEN

TYPES = list(B.QUANT_TYPES.items())


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


@pytest.mark.parametrize("name,t", TYPES)
def test_kat_quantize_fns_generator(orc, golden_ops, name, t):
    """LC/tests/test-quantize-fns.cpp:26-30,95-113 generator: quantize, dequantize, vec_dot."""
    g = golden_ops
    a, b = synthetic_cos(4096, 0.0), synthetic_cos(4096, 1.0)
    assert np.array_equal(a, g["kat_a"]) and np.array_equal(b, g["kat_b"])
    wq = orc.quantize(t, a[None, :])
    xq = orc.from_float(B.VEC_DOT_TYPE[t], b)
    assert np.array_equal(wq, g[f"kat_{name}_wq"])
    assert np.array_equal(xq, g[f"kat_{name}_xq"])
    assert np.array_equal(bits(orc.to_float(t, wq[0], 4096)), bits(g[f"kat_{name}_deq"]))
    assert bits(orc.vec_dot(t, 4096, wq[0], xq)) == bits(g[f"kat_{name}_dot"])
    # the reference's own acceptance thresholds (test-quantize-fns.cpp:16-20)
    deq = orc.to_float(t, wq[0], 4096)
    assert np.sqrt(np.sum((deq.astype(np.float64) - a) ** 2)) / 4096 < 0.002     # array_rmse(), :33-40
    assert abs(float(g[f"kat_{name}_dot"]) - float(np.dot(a.astype(np.float64), b.astype(np.float64)))) / 4096 < 0.02


@pytest.mark.parametrize("name,t", TYPES)
def test_mul_mat_golden(orc, golden_ops, name, t):
    g = golden_ops
    wq = orc.quantize(t, g["mm_w"])
    assert np.array_equal(wq, g[f"mm_{name}_wq"])
    out = orc.mul_mat(t, wq, g["mm_x"])
    assert np.array_equal(bits(out), bits(g[f"mm_{name}_out"]))


def test_row_ops_golden(orc, golden_ops):
    g = golden_ops
    assert np.array_equal(bits(orc.rms_norm(g["row_x"])), bits(g["rms_norm"]))
    assert np.array_equal(bits(orc.norm(g["row_x"])), bits(g["norm"]))
    assert np.array_equal(bits(orc.soft_max(g["softmax_x"])), bits(g["softmax"]))
    assert np.array_equal(bits(orc.silu(g["row_x"])), bits(g["silu"]))
    assert np.array_equal(bits(orc.gelu(g["row_x"])), bits(g["gelu"]))
    assert np.array_equal(bits(orc.scale_mask_soft_max(g["chain_x"], 0.125, 35)), bits(g["chain"]))


def test_fp16_luts_exhaustive(orc, golden_ops):
    g = golden_ops
    assert np.array_equal(bits(orc.silu(g["lut_in"])), bits(g["lut_silu"]))
    assert np.array_equal(bits(orc.gelu(g["lut_in"])), bits(g["lut_gelu"]))


@pytest.mark.parametrize("tag", ["llama", "llama511", "neox"])
def test_rope_golden(orc, golden_ops, tag):
    g = golden_ops
    n_past, nd, mode = (int(v) for v in g[f"rope_{tag}_p"])
    assert np.array_equal(bits(orc.rope(g[f"rope_{tag}_x"], n_past, nd, mode)), bits(g[f"rope_{tag}"]))


def _load_micro(name):
    z = np.load(os.path.join(GOLDEN, f"llama_micro_{name}.npz"))
    keys = ("n_vocab", "n_embd", "n_head", "n_head_kv", "n_layer", "n_ff", "n_rot", "n_ctx", "wtype")
    hp = dict(zip(keys, (int(v) for v in z["hp"])))
    tens = {k[2:]: z[k] for k in z.files if k.startswith("w:")}
    return z, hp, tens


@pytest.mark.parametrize("name", ["q4_0", "q5_1"])
def test_llama_micro_golden_logits(orc, name):
    z, hp, tens = _load_micro(name)
    # the weights in the fixture are what the restated quantizer produces from the same seed
    hp2, tens2 = synth.make_llama(MICRO, B.QUANT_TYPES[name], orc.quantize, seed=0x5EED0000)
    for k in tens:
        assert np.array_equal(tens[k], tens2[k]), k
    m = orc.llama(hp, tens)
    toks = z["tokens"]
    assert np.array_equal(bits(m.eval(toks[:12])), bits(z["logits_prefill"]))
    assert np.array_equal(bits(m.eval(toks[12:13])), bits(z["logits_decode"]))
    assert np.array_equal(bits(m.eval(toks[13:15])), bits(z["logits_tail"]))


# ---- against the reference's compiled ggml.c (tests/golden/reference_outputs.json) ----

def fp16_inputs():
    rng = np.random.default_rng(7)
    xs = np.concatenate([rng.standard_normal(4000).astype(np.float32) * s for s in (1e-8, 1e-6, 1e-4, 1, 300, 7e4)] +
                        [np.array([0, -0.0, 65504, 65519.9, 65520, 1e-7, 5.96e-8, 2.98e-8, 3e-8, np.inf, -np.inf], np.float32)])
    hs = np.array([h for h in range(65536) if (h & 0x7c00) != 0x7c00], np.uint16)
    return xs, hs


def test_fp16_conversions_vs_reference(orc, reference):
    xs, hs = fp16_inputs()
    reference("fp16/fp32_to_fp16", np.array([orc.lib.or_fp32_to_fp16(float(x)) for x in xs], np.uint16))
    reference("fp16/fp16_to_fp32", np.array([orc.lib.or_fp16_to_fp32(int(h)) for h in hs], np.float32))


def rows_inputs(t, K):
    rng = np.random.default_rng(K + t)
    w = (rng.standard_normal((16, K)) / np.sqrt(K)).astype(np.float32)
    x = (rng.standard_normal((3, K)) * rng.uniform(0.01, 30)).astype(np.float32)
    return w, x


@pytest.mark.parametrize("name,t", TYPES)
@pytest.mark.parametrize("K", [64, 4096, 11008])
def test_rows_vs_reference(orc, reference, name, t, K):
    w, x = rows_inputs(t, K)
    wq = orc.quantize(t, w)
    reference(f"rows/{name}/K{K}/quantize", wq)
    reference(f"rows/{name}/K{K}/from_float", orc.from_float(B.VEC_DOT_TYPE[t], x[0]))
    reference(f"rows/{name}/K{K}/mul_mat", orc.mul_mat(t, wq, x))


LLAMA_CASES = [("tiny", "q4_0"), ("tiny", "q4_1"), ("tiny", "q5_0"), ("small", "q5_1"), ("small", "q8_0")]


@pytest.mark.parametrize("cfg,name", LLAMA_CASES)
def test_llama_vs_reference(orc, reference, cfg, name):
    hp, tens = synth.make_llama(synth.CONFIGS[cfg], B.QUANT_TYPES[name], orc.quantize)
    toks = synth.make_tokens(hp, 37)
    mo = orc.llama(hp, tens)
    key = f"llama/{cfg}/{name}"
    for lo, hi in ((0, 33), (33, 34), (34, 37)):
        reference(f"{key}/eval {lo}:{hi}", mo.eval(toks[lo:hi]))
    reference(f"{key}/kv 0", mo.kv(0))
    reference(f"{key}/kv 1", mo.kv(1))
    # the reference result does not depend on the thread split nor on batching (one vec_dot per dst element): the recorded rows are its
    # single-threaded token-by-token evaluation
    mo.reset()
    reference(f"{key}/token by token 0:8", mo.eval(toks[:8]))


def test_llama_rope_overrides_and_set_n_past_vs_reference(orc, reference):
    """RoPEOverrides (op_rope_inplace -> ggml_rope_custom_inplace, crates/ggml/src/context.rs:558-590) and the position restore used
    by bench.py's CPU arm: the plain-C port and the reference's compiled ggml.c agree bit for bit."""
    hp, tens = synth.make_llama(synth.CONFIGS["tiny"], B.Q4_0, orc.quantize)
    toks = synth.make_tokens(hp, 30)
    mo = orc.llama(hp, tens)
    plain = mo.eval(toks[:9]).copy()
    mo.reset()
    mo.set_rope(26000.0, 0.5)
    b = mo.eval(toks[:20])
    reference("rope_overrides/eval 0:20", b)
    assert not np.array_equal(bits(b[:9]), bits(plain))                 # the override really changes the result
    reference("rope_overrides/eval 20:21", mo.eval(toks[20:21]))
    # rewind to position 12 (the cache rows 12.. are simply overwritten) and continue
    mo.set_n_past(12)
    reference("rope_overrides/eval 12:15 after set_n_past(12)", mo.eval(toks[12:15]))
