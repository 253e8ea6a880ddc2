"""Record what the reference's own compiled ggml.c (oracle/_ref/libggml_ref.so) returns for the seeded inputs of the tests that compare with it.

TEST INFRASTRUCTURE.  Run where oracle/_ref has been built:  python -m oracle.gen_reference_outputs [REFERENCE_CHECKOUT]
  tests/golden/reference_outputs.json   fingerprint (tests/conftest.py) of every array the tests compare bit for bit; the arrays themselves
                                        (whole-model logits, KV caches, mat-mul outputs) would not fit in the repository
  tests/golden/kquants_ref.npz          the small K-quant arrays the CPU tests take as they are (quantized rows, q8_K rows, products)
  tests/golden/reference_cuda_bindings.json   the extern fns of crates/ggml/sys/src/cuda.rs (only with REFERENCE_CHECKOUT)
The inputs and token schedules are the tests' own (imported from them), so a test and its record cannot drift apart.  Where the oracle
computes the same thing, the record is also checked against it here.
"""
import json
import os
import re
import sys

import numpy as np

from . import bindings as B
from . import synth

ROOT = os.path.dirname(B.HERE)
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, os.path.join(ROOT, "tests"))

from conftest import fingerprint  # noqa: E402
import test_gpu_kquants as TK  # noqa: E402
import test_gpu_long_context as TLC  # noqa: E402
import test_gpu_neox as TN  # noqa: E402
import test_kquants_lane_arithmetic as TL  # noqa: E402
import test_oracle_kquants as TOK  # noqa: E402
import test_oracle_pin as TP  # noqa: E402


def main():
    ref, orc = B.RefLib("ref"), B.Oracle()
    rec = {}

    def put(key, a, oracle=None):
        assert key not in rec, key
        rec[key] = fingerprint(a)
        if oracle is not None:
            assert fingerprint(oracle)["sha256"] == rec[key]["sha256"], f"{key}: the oracle disagrees with the reference"

    # ---- tests/test_oracle_pin.py
    xs, hs = TP.fp16_inputs()
    put("fp16/fp32_to_fp16", np.array([ref.lib.rh_fp32_to_fp16(float(x)) for x in xs], np.uint16))
    put("fp16/fp16_to_fp32", np.array([ref.lib.rh_fp16_to_fp32(int(h)) for h in hs], np.float32))
    for name, t in TP.TYPES:
        for K in (64, 4096, 11008):
            w, x = TP.rows_inputs(t, K)
            wq = ref.quantize(t, w)
            put(f"rows/{name}/K{K}/quantize", wq, orc.quantize(t, w))
            put(f"rows/{name}/K{K}/from_float", ref.from_float(B.VEC_DOT_TYPE[t], x[0]))
            put(f"rows/{name}/K{K}/mul_mat", ref.mul_mat(t, wq, x, n_threads=3), orc.mul_mat(t, wq, x))
    for cfg, name in TP.LLAMA_CASES:
        hp, tens = synth.make_llama(synth.CONFIGS[cfg], B.QUANT_TYPES[name], orc.quantize)
        toks = synth.make_tokens(hp, 37)
        mr = ref.llama(hp, tens, n_threads=4, n_batch=64)
        key = f"llama/{cfg}/{name}"
        for lo, hi in ((0, 33), (33, 34), (34, 37)):
            put(f"{key}/eval {lo}:{hi}", mr.eval(toks[lo:hi]))
        put(f"{key}/kv 0", mr.kv(0))
        put(f"{key}/kv 1", mr.kv(1))
        mr.close()
        mr1 = ref.llama(hp, tens, n_threads=1, n_batch=64)
        put(f"{key}/token by token 0:8", np.concatenate([mr1.eval(toks[i:i + 1]) for i in range(8)]))
        mr1.close()
    hp, tens = synth.make_llama(synth.CONFIGS["tiny"], B.Q4_0, orc.quantize)
    toks = synth.make_tokens(hp, 30)
    mr = ref.llama(hp, tens, n_threads=3, n_batch=64)
    mr.set_rope(26000.0, 0.5)
    put("rope_overrides/eval 0:20", mr.eval(toks[:20]))
    put("rope_overrides/eval 20:21", mr.eval(toks[20:21]))
    mr.set_n_past(12)
    put("rope_overrides/eval 12:15 after set_n_past(12)", mr.eval(toks[12:15]))
    mr.close()

    # ---- tests/test_gpu_kquants.py (GPU tests: recorded here, compared on the device)
    q8 = np.stack([ref.from_float(B.Q8_K, row).reshape(-1, 292) for row in TK.q8_K_inputs()])
    q8[q8[:, :, :4].copy().view(np.float32)[:, :, 0] == 0.0, 260:] = 0          # bsums the reference leaves unwritten
    put("kquant/quantize_q8_K", q8)
    for name, t in B.KQUANT_TYPES.items():
        for K, N, Bn in TK.MUL_MAT_SHAPES:
            wq, x = TK.mul_mat_inputs(t, K, N, Bn)
            put(f"kquant/mul_mat/{name}/K{K} N{N} B{Bn}", ref.mul_mat(t, wq, x))
        wq, xs = TK.seam_inputs(t)
        for x in xs:
            put(f"kquant/seam/{name}/B{x.shape[0]}", ref.mul_mat(t, wq, x))

    # ---- tests/test_gpu_neox.py
    def schedule(key, mr, toks, sched):
        for lo, hi, *last in sched:
            out = mr.eval(toks[lo:hi])
            put(f"{key}/{lo}:{hi} last row" if last else f"{key}/{lo}:{hi}", out[-1:] if last else out)
        mr.close()

    for cfg in ("par", "seq"):
        for name in ("q4_0", "q4_1", "q5_0", "q5_1", "q8_0"):
            hp, tens = synth.make_neox(TN.CFGS[cfg], B.QUANT_TYPES[name], orc.quantize)
            schedule(f"neox/{cfg}/{name}", ref.neox(hp, tens, n_threads=8, n_batch=64), synth.make_tokens(hp, 60), TN.SCHEDULES["neox"])
    for name in ("q4_0", "q5_1"):
        hp, tens = synth.make_neox(TN.NEOX_20B_2L, B.QUANT_TYPES[name], orc.quantize)
        schedule(f"neox_20b/{name}", ref.neox(hp, tens, n_threads=8, n_batch=256), synth.make_tokens(hp, 270), TN.SCHEDULES["neox_20b"])
    for name in ("q4_0", "q5_1", "q8_0"):
        for lm_head in (False, True):
            hp, tens = synth.make_gpt2(TN.GPT2_CFG, B.QUANT_TYPES[name], orc.quantize, lm_head=lm_head)
            schedule(f"gpt2/{name}/lm_head={lm_head}", ref.gpt2(hp, tens, n_threads=8, n_batch=64), synth.make_tokens(hp, 60), TN.SCHEDULES["gpt2"])
    hp, tens = synth.make_gpt2(TN.GPT2_117M_3L, B.Q4_0, orc.quantize)
    schedule("gpt2_117m", ref.gpt2(hp, tens, n_threads=8, n_batch=64), synth.make_tokens(hp, 40), TN.SCHEDULES["gpt2_117m"])

    # ---- tests/test_gpu_long_context.py
    hp, tens = synth.make_neox(TLC.NEOX_LONG_CFG, B.Q4_0, orc.quantize)
    schedule("neox_long/par/q4_0", ref.neox(hp, tens, n_threads=8, n_batch=512), synth.make_tokens(hp, 4096), TLC.LONG_CTX_SCHEDULE)
    hp, tens = synth.make_gpt2(TLC.GPT2_LONG_CFG, B.Q8_0, orc.quantize)
    schedule("gpt2_long/q8_0", ref.gpt2(hp, tens, n_threads=8, n_batch=512), synth.make_tokens(hp, 4096), TLC.LONG_CTX_SCHEDULE)

    with open(os.path.join(GOLDEN, "reference_outputs.json"), "w") as f:
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(v)}" for k, v in sorted(rec.items())) + "\n}\n")

    # ---- tests/test_oracle_kquants.py, tests/test_kquants_lane_arithmetic.py
    kq = {}
    _, x, w = TOK._inputs()
    for b in range(x.shape[0]):
        q = ref.from_float(B.Q8_K, x[b]).reshape(-1, 292)
        q[q[:, :4].copy().view(np.float32)[:, 0] == 0.0, 260:] = 0
        kq[f"q8_K_row{b}"] = q.reshape(-1)
    _, wl = TL.lane_inputs()
    for name, t in B.KQUANT_TYPES.items():
        kq[f"{name}_wq"] = np.stack([ref.from_float(t, r) for r in w])
        kq[f"{name}_mul_mat"] = ref.mul_mat(t, kq[f"{name}_wq"], x)
        kq[f"lane_{name}_wq"] = np.stack([ref.from_float(t, r) for r in wl])
    np.savez_compressed(os.path.join(GOLDEN, "kquants_ref.npz"), **kq)

    if len(sys.argv) > 1:
        src = open(os.path.join(sys.argv[1], "crates", "ggml", "sys", "src", "cuda.rs")).read()
        with open(os.path.join(GOLDEN, "reference_cuda_bindings.json"), "w") as f:
            json.dump(sorted(re.findall(r"pub fn (\w+)\(", src)), f, indent=0)
            f.write("\n")
    for f in ("reference_outputs.json", "kquants_ref.npz", "reference_cuda_bindings.json"):
        print(f, os.path.getsize(os.path.join(GOLDEN, f)))


if __name__ == "__main__":
    main()
