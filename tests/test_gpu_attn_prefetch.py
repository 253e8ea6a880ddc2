"""The fused decode attention loads the cached K rows and V columns below n_past before it waits for the QKV launch
(B200_ATTN_PREFETCH=1, the default) or after it (=0).  Both orders decode bit-exact against the oracle at contexts that need more
than one pass of K rows per CTA (n_kv > 1024 at head size 128, > 512 at 64), and right after a rewind, where the cache above n_past
holds the rows of the abandoned tokens.  The switch is read once per process, so each order runs in a process of its own."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:            # also run as a script: the worker of one order
    sys.path.insert(0, ROOT)

from oracle import bindings as B    # noqa: E402
from oracle import synth            # noqa: E402

pytestmark = pytest.mark.gpu

# shapes the fused decode graph serves (n_rot = head size, n_ff % 256 == 0), small enough for the CPU oracle at n_ctx 2048
GEOMETRIES = {
    "hd128": dict(synth.CONFIGS["gqa8"], n_head=4, n_head_kv=4, n_rot=128, n_ctx=2048),
    "hd64": dict(synth.CONFIGS["gqa8"], n_head_kv=8, n_ctx=2048),
    "hd64-gqa": dict(synth.CONFIGS["gqa8"], n_ctx=2048),
}
REWIND = 1500           # not a multiple of 8: the V chunk holding column n_past also holds stale columns


def schedule():
    """(kind, tokens a..b or rewind target) in order: batches in chunks of at most 512, single-token decode steps across both pass edges"""
    steps = [("batch", 0, 512), ("batch", 512, 1022)]
    steps += [("decode", i, i + 1) for i in range(1022, 1028)]
    steps += [("batch", 1028, 1540), ("batch", 1540, 2044)]
    steps += [("decode", i, i + 1) for i in range(2044, 2048)]
    steps += [("rewind", REWIND, None), ("decode", REWIND, REWIND + 1)]
    return steps


def model(orc, geom):
    hp, tens = synth.make_llama(GEOMETRIES[geom], B.Q4_0, orc.quantize)
    return hp, tens, synth.make_tokens(hp, 2048)


def run_native(geom, out):
    """worker: the decode logits of every step of schedule() and both caches, into the npz `out`"""
    import llm_b200
    orc = B.Oracle()
    hp, tens, toks = model(orc, geom)
    m = llm_b200.Llama(hp, llm_b200.ModelParameters(context_size=hp["n_ctx"]), tens)
    s = m.start_session(llm_b200.InferenceSessionConfig(n_batch=512))
    res = {}
    for kind, a, b in schedule():
        if kind == "rewind":
            s.rewind(a)
            continue
        g = s.evaluate(toks[a:b], all_logits=kind == "decode")
        if kind == "decode":
            assert s.last_launches == 7 * hp["n_layer"] + 3, ("fused decode graph not used", s.last_launches)
            res[f"decode{a}"] = g
    res["kv0"], res["kv1"] = s.kv(0), s.kv(1)
    np.savez(out, **res)
    s.close(); m.close()


@pytest.mark.slow
@pytest.mark.parametrize("geom", list(GEOMETRIES))
def test_attn_prefetch_bit_exact_past_one_pass(orc, geom, tmp_path):
    got = {}
    for pf in ("1", "0"):
        out = str(tmp_path / f"pf{pf}.npz")
        env = dict(os.environ, B200_ATTN_PREFETCH=pf)
        py = [sys.executable] + (["-s"] if sys.flags.no_user_site else [])
        r = subprocess.run(py + [os.path.abspath(__file__), geom, out], cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, (pf, r.stdout[-2000:], r.stderr[-4000:])
        got[pf] = np.load(out)
    hp, tens, toks = model(orc, geom)
    mo = orc.llama(hp, tens)
    for kind, a, b in schedule():
        if kind == "rewind":
            mo.set_n_past(a)
            continue
        want = mo.eval(toks[a:b])
        if kind == "decode":
            for pf, g in got.items():
                d = g[f"decode{a}"]
                assert np.array_equal(d.view(np.uint32), want.view(np.uint32)), (geom, f"B200_ATTN_PREFETCH={pf}", f"decode at n_past={a}",
                                                                                  float(np.abs(d - want).max()))
    for which in (0, 1):
        ref = mo.kv(which)
        for pf, g in got.items():
            a = g[f"kv{which}"]
            assert np.array_equal(a, ref[:a.size]), (geom, f"B200_ATTN_PREFETCH={pf}", which)
    mo.close()


if __name__ == "__main__":
    run_native(sys.argv[1], sys.argv[2])
