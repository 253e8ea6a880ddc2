"""Decode past 3072 cached positions.  The cluster attention of the fused decode schedules holds a whole context bucket (scores, probabilities and
the head's V rows) in one CTA's shared memory; buckets are multiples of 256 capped at n_ctx, and the largest that fits is 3072 (3264 when it is
the capped last bucket).  So with context_size > 3264 every token past position 3072 decodes through another path:
  LLaMA              the two-kernel attention attn_kq + attn_sv: 8 launches per layer instead of 7
  GPT-NeoX / GPT-2   the per-op schedule, node by node
  tensor parallel    no other path (the exchange lives in the cluster attention's epilogue): start_session refuses such a context_size
The two-kernel attention also runs at every length with B200_ATTN_FUSED=0, which is how its quantize epilogue is covered for every block format
at short contexts.  That switch is read once per process, so those cases run in a process of their own."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:            # also run as a script: the worker of the B200_ATTN_FUSED=0 cases
    sys.path.insert(0, ROOT)

from oracle import bindings as B    # noqa: E402
from oracle import synth            # noqa: E402
from test_gpu_neox import CFGS as NEOX_CFGS, GPT2_CFG, check   # noqa: E402

pytestmark = pytest.mark.gpu

FUSED_MAX = 3072        # the largest n_kv whose bucket the cluster attention holds when n_ctx > 3264


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def chunks(lo, hi, size=512):
    return [(a, min(a + size, hi)) for a in range(lo, hi, size)]


# ---- a. LLaMA past the switch, against the oracle ------------------------------------------------------------------------------------------
# the geometries of test_gpu_attn_prefetch.py (n_ctx a multiple of 128, as the decode graph requires); at 3968 the last bucket is capped at
# n_ctx and is not a multiple of 256
LONG_GEOMETRIES = {
    "hd128": dict(synth.CONFIGS["gqa8"], n_head=4, n_head_kv=4, n_rot=128, n_ctx=4096),
    "hd64": dict(synth.CONFIGS["gqa8"], n_head_kv=8, n_ctx=4096),
    "hd64-gqa": dict(synth.CONFIGS["gqa8"], n_ctx=4096),
    "hd64-gqa-ctx3968": dict(synth.CONFIGS["gqa8"], n_ctx=3968),
}


def long_schedule(n_ctx):
    """(kind, a, b) in order: batches of at most 512, single decode steps across the 3072 -> 3328 bucket edge and in the last bucket
    (n_kv = n_ctx), a step at a full context, then rewinds onto stale cache rows past the switch (3500: the V chunk holding column n_past also
    holds stale columns) and before it (3000: back on the cluster attention, whose graph is already captured)"""
    steps = [("batch", a, b) for a, b in chunks(0, 3068)]
    steps += [("decode", i, i + 1) for i in range(3068, 3077)]
    steps += [("batch", a, b) for a, b in chunks(3077, n_ctx - 8)]
    steps += [("decode", i, i + 1) for i in range(n_ctx - 8, n_ctx)]
    steps += [("full", n_ctx, None)]
    for r in (3500, 3000):
        steps += [("rewind", r, None), ("decode", r, r + 1), ("decode", r + 1, r + 2)]
    return steps


def llama_launches(n_layer, n_kv):
    return (7 if n_kv <= FUSED_MAX else 8) * n_layer + 3


@pytest.mark.slow
@pytest.mark.parametrize("geom", list(LONG_GEOMETRIES))
def test_llama_decode_past_cluster_attention(orc, geom):
    import llm_b200
    hp, tens = synth.make_llama(LONG_GEOMETRIES[geom], B.Q4_0, orc.quantize)
    n_ctx, n_layer = hp["n_ctx"], hp["n_layer"]
    toks = synth.make_tokens(hp, n_ctx)
    m = llm_b200.Llama(hp, llm_b200.ModelParameters(context_size=n_ctx), tens)
    s = m.start_session(llm_b200.InferenceSessionConfig(n_batch=512))
    mo = orc.llama(hp, tens)
    for kind, a, b in long_schedule(n_ctx):
        if kind == "rewind":
            s.rewind(a); mo.set_n_past(a)
            continue
        if kind == "full":
            assert s.n_past == n_ctx
            with pytest.raises(llm_b200.ContextFull):
                s.evaluate(toks[:1])
            continue
        g = s.evaluate(toks[a:b], all_logits=True)
        if kind == "decode":
            assert s.last_launches == llama_launches(n_layer, b), (geom, f"decode at n_past={a}", s.last_launches)
        want = mo.eval(toks[a:b])
        assert same_bits(g, want), (geom, f"{kind} {a}:{b}", float(np.abs(g - want).max()))
    for which in (0, 1):
        got = s.kv(which)
        assert np.array_equal(got, mo.kv(which)[:got.size]), (geom, which)
    mo.close(); s.close(); m.close()


# ---- b. the two-kernel attention for every block format at short contexts (B200_ATTN_FUSED=0) ----------------------------------------------
SHORT_CFGS = dict(synth.CONFIGS, **{"gqa8-hd128": dict(synth.CONFIGS["gqa8"], n_head=4, n_head_kv=4, n_rot=128)})
SHORT_CASES = [("tiny8", "q4_0"), ("tiny8", "q4_1"), ("tiny8", "q5_0"), ("tiny8", "q5_1"), ("tiny8", "q8_0"), ("gqa8", "q4_0"), ("gqa8", "q5_1"),
               ("gqa8-hd128", "q4_0")]


def short_schedule():
    """the schedule of test_gpu_llama.py::test_decode_kernel_bit_exact: prefill, 40 decode steps, a rewind, a batch, a step after it"""
    steps = [("batch", 0, 21)] + [("decode", i, i + 1) for i in range(21, 61)]
    return steps + [("rewind", 30, None), ("decode", 30, 31), ("batch", 31, 35), ("decode", 35, 36)]


def short_model(orc, cfg, name):
    hp, tens = synth.make_llama(SHORT_CFGS[cfg], B.QUANT_TYPES[name], orc.quantize)
    return hp, tens, synth.make_tokens(hp, 70)


def run_two_kernel(cfg, name, out):
    """worker: the logits and launch count of every step of short_schedule() and both caches, into the npz `out`"""
    import llm_b200
    hp, tens, toks = short_model(B.Oracle(), cfg, name)
    m = llm_b200.Llama(hp, llm_b200.ModelParameters(context_size=hp["n_ctx"]), tens)
    s = m.start_session(llm_b200.InferenceSessionConfig(n_batch=64))
    res = {}
    for i, (kind, a, b) in enumerate(short_schedule()):
        if kind == "rewind":
            s.rewind(a)
            continue
        res[f"logits{i}"] = s.evaluate(toks[a:b], all_logits=True)
        res[f"launches{i}"] = np.int32(s.last_launches)
    res["kv0"], res["kv1"] = s.kv(0), s.kv(1)
    np.savez(out, **res)
    s.close(); m.close()


@pytest.mark.parametrize("cfg,name", SHORT_CASES)
def test_two_kernel_attention_bit_exact(orc, cfg, name, tmp_path):
    out = str(tmp_path / "two_kernel.npz")
    env = dict(os.environ, B200_ATTN_FUSED="0")
    py = [sys.executable] + (["-s"] if sys.flags.no_user_site else [])
    r = subprocess.run(py + [os.path.abspath(__file__), cfg, name, out], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
    got = np.load(out)
    hp, tens, toks = short_model(orc, cfg, name)
    mo = orc.llama(hp, tens)
    for i, (kind, a, b) in enumerate(short_schedule()):
        if kind == "rewind":
            mo.set_n_past(a)
            continue
        want, g = mo.eval(toks[a:b]), got[f"logits{i}"]
        assert same_bits(g, want), (cfg, name, f"{kind} {a}:{b}", float(np.abs(g - want).max()))
        if kind == "decode":
            assert int(got[f"launches{i}"]) == 8 * hp["n_layer"] + 3, ("two-kernel decode graph not used", a, int(got[f"launches{i}"]))
    for which in (0, 1):
        a = got[f"kv{which}"]
        assert np.array_equal(a, mo.kv(which)[:a.size]), (cfg, name, which)
    mo.close()


# ---- c. GPT-NeoX and GPT-2 at context_size 4096, against the recorded reference -------------------------------------------------------------
# oracle/gen_reference_outputs.py records what the reference returns for these configs and schedules
NEOX_LONG_CFG = dict(NEOX_CFGS["par"], n_ctx=4096)
GPT2_LONG_CFG = dict(GPT2_CFG, n_ctx=4096)            # 4096 rows of wpe
LONG_CTX_SCHEDULE = (chunks(0, 3068) + [(i, i + 1) for i in range(3068, 3077)] + chunks(3077, 4088) + [(i, i + 1) for i in range(4088, 4096)])


@pytest.mark.parametrize("arch", ["neox", "gpt2"])
def test_neox_gpt2_decode_past_cluster_attention(orc, reference, arch):
    """single tokens up to n_kv 3072 run the fused graph; past it they run node by node; every chunk is bit-identical to the reference"""
    from llm_b200.neox import Gpt2, GptNeoX
    if arch == "neox":
        hp, tens = synth.make_neox(NEOX_LONG_CFG, B.Q4_0, orc.quantize)
        m, key, fused = GptNeoX(hp, tens), "neox_long/par/q4_0", 8 * hp["n_layer"] + 3
    else:
        hp, tens = synth.make_gpt2(GPT2_LONG_CFG, B.Q8_0, orc.quantize)
        m, key, fused = Gpt2(hp, tens), "gpt2_long/q8_0", 8 * hp["n_layer"] + 4
    toks = synth.make_tokens(hp, 4096)
    s = m.start_session(512)
    for lo, hi in LONG_CTX_SCHEDULE:
        check(reference, key, lo, hi, s.evaluate(toks[lo:hi], all_logits=True))
        if hi - lo == 1:
            if hi <= FUSED_MAX:
                assert s.last_launches == fused, ("fused decode schedule not used", lo, s.last_launches)
            else:
                assert s.last_launches > fused, ("per-op schedule not used", lo, s.last_launches)
    s.close(); m.close()


# ---- d. tensor parallel: a context_size the cluster attention cannot hold is refused at start_session --------------------------------------
TP_CFG = dict(n_vocab=1024, n_embd=512, n_head=8, n_head_kv=8, n_layer=2, n_ff=1024, n_rot=64)


def test_tensor_parallel_refuses_context_past_cluster_attention(orc, capfd):
    """a shard's session is set up before its peers are connected, so one GPU is enough to see rank 0 of 2 accept or refuse it"""
    import llm_b200
    from llm_b200 import tp
    cfg = llm_b200.InferenceSessionConfig(n_batch=8)
    hp, tens = synth.make_llama(dict(TP_CFG, n_ctx=4096), B.Q4_0, orc.quantize)
    for n_ctx, ok in ((3264, True), (4096, False)):
        m = tp.TpLlama(hp, llm_b200.ModelParameters(context_size=n_ctx), tens, rank=0, world=2, device=0)
        capfd.readouterr()
        if ok:
            llm_b200.InferenceSession(m, cfg).close()
        else:
            with pytest.raises(RuntimeError):
                llm_b200.InferenceSession(m, cfg)
            assert f"context_size {n_ctx}" in capfd.readouterr().err
        m.close()


if __name__ == "__main__":
    run_two_kernel(*sys.argv[1:4])
