"""Per-launch timeline of the graph decode schedule (tuning aid): python tools/decode_timeline.py [n_layer]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))   # run from anywhere: the repo root holds llm_b200/ and oracle/

import ctypes as C, os, sys
import numpy as np
os.environ["B200_DECODE_PROF"] = "1"
import llm_b200
from llm_b200 import _lib
L = _lib.lib()
nl = int(sys.argv[1]) if len(sys.argv) > 1 else 32
hp = dict(n_vocab=32000, n_embd=4096, n_head=32, n_head_kv=32, n_layer=nl, n_rot=128, n_ff=11008, wtype=2)
m = llm_b200.Llama(hp, llm_b200.ModelParameters(context_size=2048)); m.synthesize(1)
s = m.start_session(llm_b200.InferenceSessionConfig(n_batch=512))
toks = np.random.default_rng(0).integers(0, 32000, 520, dtype=np.int32)
s.evaluate(toks[:512])
for i in range(5):
    s.evaluate(toks[512 + i:513 + i])
per_layer = ["norm", "qkv", "attn", "wo", "norm2", "w13", "w2"] if os.environ.get("B200_ATTN_FUSED", "1") != "0" else ["norm", "qkv", "kq", "sv", "wo", "norm2", "w13", "w2"]
n = len(per_layer) * nl + 3
L.b200_session_decode_timeline(s._s, None, 0, 1)
s.evaluate(toks[517:518])
buf = (C.c_ulonglong * (9 * n))()
L.b200_session_decode_timeline(s._s, buf, n, 0)
t = np.array(buf[:], dtype=np.float64).reshape(9, n)
beg, end, rdy, begx, rdyx, ff, ffx, lf, sm = t
names = ["embed"] + per_layer * nl + ["normF", "logits"]
t0 = beg[1]
print("token span %.1f us (first norm begin -> logits end)" % ((end[-1] - t0) / 1e3))
agg = {}
prev_end = None
def rel(a, i): return (a[i] - beg[i]) / 1e3 if 0 < a[i] < 1e19 else float("nan")
for i in range(1, n):
    dur = (end[i] - beg[i]) / 1e3
    gap = (beg[i] - prev_end) / 1e3 if prev_end is not None else 0.0
    prev_end = end[i]
    vals = [dur, gap, rel(begx, i), rel(rdy, i), rel(rdyx, i), rel(ff, i), rel(ffx, i), rel(lf, i)]
    a = agg.setdefault(names[i], [0] + [0.0] * len(vals)); a[0] += 1
    for k, v in enumerate(vals): a[k + 1] += 0.0 if v != v else v
print("per kernel type, mean us relative to the first CTA's start: dur | gap before | last CTA start | x ready first/last | first stage landed first/last CTA | last stage landed")
tot_d = tot_g = 0.0
for k, a in agg.items():
    c = a[0]; v = [x / c for x in a[1:]]
    print(f"  {k:7s} n={c:3d} dur {v[0]:6.2f} gap {v[1]:5.2f} | lastCTA {v[2]:5.2f} | xready {v[3]:5.2f}/{v[4]:5.2f} | stage0 {v[5]:5.2f}/{v[6]:5.2f} | laststage {v[7]:6.2f} | total {(a[1]+a[2])/1e3:6.3f} ms")
    tot_d += a[1]; tot_g += a[2]
print(f"sum durations {tot_d/1e3:.3f} ms, sum gaps {tot_g/1e3:.3f} ms")
# the fused attention's phases (decode_ops.cu attn_fused_kernel), mean us relative to the first CTA's start; the QKV launch before it is the
# one its pdl_wait waits for
ia = [i for i in range(1, n) if names[i] == "attn"]
if ia:
    m = lambda a, idx=None: float(np.nanmean([rel(a, i) if idx is None else (a[idx(i)] - beg[i]) / 1e3 for i in ia]))
    print("attn phases, mean us relative to the first CTA's start (first/last CTA):")
    print(f"  lastCTA start {m(begx):5.2f} | qkv end {m(end, lambda i: i - 1):5.2f} | past pdl_wait {m(rdy):5.2f}/{m(rdyx):5.2f} | "
          f"KQ share done {m(ff):5.2f}/{m(ffx):5.2f} | scores exchanged {m(lf):5.2f} | soft_max done {m(sm):5.2f} | end {m(end):5.2f}")
