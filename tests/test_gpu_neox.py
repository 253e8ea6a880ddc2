"""Native GPT-NeoX runtime (llm_b200/csrc/neox.cu + the fused decode schedule of decode_ops.cu) against the reference's own ggml CPU build running the
reference's GPT-NeoX graph (oracle/ref_gpt2.c): logits bit-identical for prefill, the CUDA-graph decode steps, batches after decode,
parallel and sequential residual, all five block formats, and the NeoX-20B head geometry (head size 96, n_rot 24).  What the reference returned
for these models and token chunks is recorded in tests/golden/reference_outputs.json (oracle/gen_reference_outputs.py evaluates the same
SCHEDULES on the reference)."""
import numpy as np
import pytest

from oracle import bindings as B
from oracle import synth

pytestmark = pytest.mark.gpu


def check(reference, key, lo, hi, got):
    reference(f"{key}/{lo}:{hi}", np.asarray(got, np.float32))


CFGS = {   # K = 256 (8 quant blocks: the streaming mat-vec's granularity), head sizes 64 / 32, rotary dims < and == head size, both residual forms
    "par": dict(n_vocab=384, n_ctx=128, n_embd=256, n_head=4, n_layer=2, n_rot=16, use_parallel_residual=1),
    "seq": dict(n_vocab=384, n_ctx=128, n_embd=256, n_head=8, n_layer=2, n_rot=32, use_parallel_residual=0),
}
NEOX_20B_2L = dict(synth.NEOX_CONFIGS["neox-20b"], n_layer=2, n_ctx=512)
GPT2_CFG = dict(n_vocab=320, n_ctx=128, n_embd=256, n_head=4, n_layer=2)
GPT2_117M_3L = dict(synth.GPT2_CONFIGS["gpt2-117m"], n_layer=3)
# token chunks (lo, hi) evaluated in order; a chunk of the form (lo, hi, "last") asks for the last row's logits only
SCHEDULES = {
    "neox": [(0, 20)] + [(i, i + 1) for i in range(20, 30)] + [(30, 47), (47, 48), (48, 52, "last")],
    "neox_20b": [(0, 130)] + [(i, i + 1) for i in range(130, 134)] + [(134, 254)] + [(i, i + 1) for i in range(254, 259)],
    "gpt2": [(0, 20)] + [(i, i + 1) for i in range(20, 28)] + [(28, 45), (45, 46)],
    "gpt2_117m": [(0, 32)] + [(i, i + 1) for i in range(32, 36)],
}


def run_schedule(reference, key, s, toks, schedule, decode_launches, decode_range):
    """evaluate the chunks on the native session; single-token steps inside decode_range must run the fused decode schedule"""
    for lo, hi, *last in schedule:
        if last:
            check(reference, key, lo, f"{hi} last row", s.evaluate(toks[lo:hi]))
            continue
        check(reference, key, lo, hi, s.evaluate(toks[lo:hi], all_logits=True))
        if hi - lo == 1 and decode_range[0] <= lo < decode_range[1]:
            assert s.last_launches == decode_launches, ("fused decode schedule not used", s.last_launches)


@pytest.mark.parametrize("name", ["q4_0", "q4_1", "q5_0", "q5_1", "q8_0"])
@pytest.mark.parametrize("cfg", ["par", "seq"])
def test_neox_native_vs_reference(orc, reference, cfg, name):
    from llm_b200.neox import GptNeoX
    hp, tens = synth.make_neox(CFGS[cfg], B.QUANT_TYPES[name], orc.quantize)
    toks = synth.make_tokens(hp, 60)
    m = GptNeoX(hp, tens)
    s = m.start_session(64)
    run_schedule(reference, f"neox/{cfg}/{name}", s, toks, SCHEDULES["neox"], 8 * hp["n_layer"] + 3, (20, 30))
    s.close(); m.close()


@pytest.mark.slow
@pytest.mark.parametrize("name", ["q4_0", "q5_1"])
def test_neox_20b_geometry_two_layers(orc, reference, name):
    """BASELINE.json configs[4] geometry: n_embd 6144, 64 heads of 96, n_rot 24, vocab 50432, parallel residual; 2 layers.
    Prefill 130 tokens (tcgen05 GEMM path, batch >= 96) + decode steps across the 256 bucket edge."""
    from llm_b200.neox import GptNeoX
    hp, tens = synth.make_neox(NEOX_20B_2L, B.QUANT_TYPES[name], orc.quantize)
    toks = synth.make_tokens(hp, 270)
    m = GptNeoX(hp, tens)
    s = m.start_session(256)
    run_schedule(reference, f"neox_20b/{name}", s, toks, SCHEDULES["neox_20b"], 8 * hp["n_layer"] + 3, (130, 134))
    s.close(); m.close()


@pytest.mark.parametrize("name", ["q4_0", "q5_1", "q8_0"])
@pytest.mark.parametrize("lm_head", [False, True])
def test_gpt2_native_vs_reference(orc, reference, name, lm_head):
    """GPT-2 (BASELINE.json configs[0] family) on the same native runtime: learned positions, c_attn in thirds, no RoPE, sequential residual, output
    projection tied to wte or a separate lm_head -- logits bit-identical to the reference's GPT-2 graph on its own ggml CPU build"""
    from llm_b200.neox import Gpt2
    hp, tens = synth.make_gpt2(GPT2_CFG, B.QUANT_TYPES[name], orc.quantize, lm_head=lm_head)
    toks = synth.make_tokens(hp, 60)
    m = Gpt2(hp, tens)
    s = m.start_session(64)
    run_schedule(reference, f"gpt2/{name}/lm_head={lm_head}", s, toks, SCHEDULES["gpt2"], 8 * hp["n_layer"] + 4, (20, 28))
    s.close(); m.close()


@pytest.mark.slow
def test_gpt2_117m_geometry(orc, reference):
    """BASELINE.json configs[0]: GPT-2 117M geometry (768 / 12 heads / 12 layers / vocab 50257 / n_ctx 1024) Q4_0, 32-token prompt + 4 decode steps"""
    from llm_b200.neox import Gpt2
    hp, tens = synth.make_gpt2(GPT2_117M_3L, B.Q4_0, orc.quantize)
    toks = synth.make_tokens(hp, 40)
    m = Gpt2(hp, tens)
    s = m.start_session(64)
    run_schedule(reference, "gpt2_117m", s, toks, SCHEDULES["gpt2_117m"], None, (0, 0))
    s.close(); m.close()
