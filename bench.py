#!/usr/bin/env python
"""bench.py -- LLaMA-7B Q4_0 tokens/sec on B200 (BASELINE.json metric): decode@1 (default line) and prefill@512 (--metric prefill).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--metric decode|prefill]    our arm (N>1: torchrun, one replica per GPU)
  python bench.py ... --dump-outputs DIR                                          also write the logits of the last timed step as DIR/*.npy
  python bench.py --impl reference [--metric decode|prefill] [...]                  the reference's own ggml CPU path, FULL 32-layer model

A "step" is one pass of the hot path over one batch: one decode token (Llama::evaluate with 1 token) at n_past = 512 on a
synthetic, device-generated LLaMA-7B Q4_0 model (BASELINE.json configs[1]).  Every headline number is measured on the CONFORMANT
path: kernels that reproduce the reference's AVX2 operation order, logits bit-identical to the reference CPU path (DESIGN.md §2).
The order-free kernels (B200_SESSION_FAST) are reported beside it under "fast_mode" and labelled non-conformant.  `value` is measured with inputs resident in
HBM (token id and logits stay on the device); `e2e` goes through the host-buffer call (b200_session_evaluate: token H2D,
logits D2H, sync) every step.  Timing: CUDA events on the backend's stream, W >= 3 warm-up steps, the 3.7 GB of weights
are far larger than the 126 MB L2 so every step streams them from HBM.  Multi-GPU (the path does not need to shard: 7B fits
one GPU) = N independent replicas, no data-path collective, "scaling": "weak".
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HP_7B = dict(n_vocab=32000, n_embd=4096, n_head=32, n_head_kv=32, n_layer=32, n_rot=128, n_ff=11008, wtype=2)
N_PAST = 512
METRIC = "LLaMA-7B Q4_0 tokens/sec (decode@1, n_past=512)"
METRIC_PREFILL = "LLaMA-7B Q4_0 tokens/sec (prefill@512)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=j["hbm_gbs"], bf16_tflops=j["bf16_tflops"], bf16_sustained=j.get("bf16_tflops_sustained", j["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source="fallback")


def algorithmic_bytes_per_token(hp, n_past, blk=18):
    """SURVEY.md §8(d): every weight byte once + the f16 KV cache read + one embedding row."""
    e, f, v, nl = hp["n_embd"], hp["n_ff"], hp["n_vocab"], hp["n_layer"]
    gqa = e // (hp["n_head"] // hp["n_head_kv"])
    per_layer = (e * e * 2 + 2 * gqa * e + 3 * e * f) // 32 * blk
    weights = nl * per_layer + v * e // 32 * blk
    kv = 2 * nl * (n_past + 1) * gqa * 2
    return weights, kv, e // 32 * blk


def prefill_flops(hp, n):
    e, f, v, nl = hp["n_embd"], hp["n_ff"], hp["n_vocab"], hp["n_layer"]
    gqa = e // (hp["n_head"] // hp["n_head_kv"])
    return 2.0 * n * (nl * (e * e * 2 + 2 * gqa * e + 3 * e * f) + v * e)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.12)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def hold(self, burst, agree=None, min_samples=2, max_s=4.0):
        """Keep the SAME load running (untimed bursts) until nvidia-smi has reported at least `min_samples` rows: its start-up (0.1 - 0.6 s on an 8-GPU
        box) can exceed a 64-token timed region, and a line without clocks is worthless.  `agree` = max over ranks, so every rank runs the same bursts."""
        if not self.proc:
            return
        t0 = time.perf_counter()
        while True:
            need = 1.0 if (len(self.rows) < min_samples and time.perf_counter() - t0 < max_s) else 0.0
            if agree is not None:
                need = agree(need)
            if need <= 0:
                break
            burst()

    def summary(self):
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# --------------------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own ggml.c (oracle/_ref, else the plain-C port) on the host cores, on the FULL model
# --------------------------------------------------------------------------------------------------------------------------------
def cpu_reference(metric, steps, warmup, log=lambda *a: None, weights=None, gpu=None, n_layer=32, budget_s=240.0):
    """The reference's ggml CPU path on the published configuration: the full `n_layer`-layer LLaMA-7B Q4_0 model (3.7 GB of blocks).

    weights = None : blocks drawn directly (oracle/synth.make_llama_random_blocks; timing does not depend on the values) -- `--impl reference`.
    weights = dict : the GPU arm's device-synthesised tensors read back (b200_model_read_tensor): the SAME model on both sides, and with
                     gpu = dict(kv=(K, V), token=id, logits=row, n_past=512) the first CPU decode step is compared bit for bit with the
                     GPU's logits at the same position (the cache contents are installed from the GPU session, so no 30 s CPU prefill).
    decode : warmup + steps single-token evaluates at n_past = 512 (position restored before every step, like the GPU arm's rewind),
             median, for several thread counts on the one loaded model -- the reference is credited with its best.
    prefill: one 512-token evaluate from an empty session per thread count (the reference computes the lm_head on all 512 rows)."""
    from oracle import bindings as B
    from oracle import synth
    kind = "reference" if B.have_ref("ref") else "port"
    nproc = os.cpu_count() or 1
    hp = dict(synth.CONFIGS["7b"], n_layer=n_layer, n_ctx=2048 if gpu else N_PAST + 64, wtype=B.Q4_0)
    t0 = time.time()
    if weights is None:
        hp, weights = synth.make_llama_random_blocks(hp, B.Q4_0)
    log(f"cpu: {n_layer}-layer LLaMA-7B Q4_0 model ready in {time.time() - t0:.1f}s ({sum(v.nbytes for v in weights.values()) / 1e9:.2f} GB)")
    t0 = time.time()
    if kind == "reference":
        m = B.RefLib("ref").llama(hp, weights, n_threads=max(1, nproc // 2), n_batch=N_PAST)
        cands = sorted({max(1, nproc // 2), min(16, nproc), min(32, nproc)}, reverse=True)
    else:
        m = B.Oracle().llama(hp, weights)
        cands = [nproc]
    log(f"cpu[{kind}]: model loaded in {time.time() - t0:.1f}s; host has {nproc} logical cores; thread counts to try: {cands}")
    toks = synth.make_tokens(hp, N_PAST + 1) if gpu is None else None
    t_start = time.time()
    out = dict(kind=kind, unit="tokens/s", parity=None)

    def set_threads(nt):
        if kind == "reference":
            m.set_threads(nt)
        else:
            os.environ["OMP_NUM_THREADS"] = str(nt)

    if metric == "prefill":
        best = None
        for nt in cands[:2]:
            set_threads(nt)
            m.set_n_past(0)
            t0 = time.time()
            m.eval(toks[:N_PAST])
            dt = time.time() - t0
            log(f"cpu[{kind}] threads={nt}: prefill@512 {dt:.2f} s")
            if best is None or dt < best[0]:
                best = (dt, nt)
            if time.time() - t_start > budget_s:
                break
        out.update(value=N_PAST / best[0], cores=best[1], ms_per_step=best[0] * 1e3,
                   sample=f"full {n_layer}-layer LLaMA-7B Q4_0, one 512-token evaluate from an empty session (lm_head on all 512 rows, as the reference does), best of {len(cands[:2])} thread counts; host has {nproc} logical cores")
        m.close()
        return out

    # ---- decode ----
    one = None
    if gpu is not None:                                        # install the GPU session's KV cache: same model, same state, same token
        for which in (0, 1):
            dst, nbytes = m.kv_ptr(which)
            src = gpu["kv"][which]
            assert src.nbytes <= nbytes, (src.nbytes, nbytes)
            C.memmove(dst, src.ctypes.data, src.nbytes)
        one = np.array([gpu["token"]], np.int32)
    else:
        set_threads(cands[0])
        t0 = time.time()
        m.eval(toks[:N_PAST])                                  # a real prefill fills the cache
        out["prefill_ms"] = (time.time() - t0) * 1e3
        log(f"cpu[{kind}] threads={cands[0]}: prefill@512 {out['prefill_ms'] / 1e3:.2f} s (fills the KV cache)")
        one = toks[N_PAST:N_PAST + 1]
    logits = np.empty((1, hp["n_vocab"]), np.float32)
    if gpu is not None:
        set_threads(cands[0])
        m.set_n_past(gpu["n_past"])
        m.eval_into(one, logits)
        same = np.array_equal(logits[0].view(np.uint32), gpu["logits"].view(np.uint32))
        out["parity"] = {"checked": f"decode step at n_past={gpu['n_past']}, full {n_layer}-layer model, device-synthesised weights read back, KV cache installed from the GPU session",
                         "bit_identical": bool(same), "max_abs_diff": float(np.abs(logits[0] - gpu["logits"]).max())}
        log(f"parity at the published configuration: logits bit-identical = {same}")
    best = None
    for nt in cands:
        set_threads(nt)
        ts = []
        for i in range(warmup + steps):
            m.set_n_past(N_PAST)
            t0 = time.time()
            m.eval_into(one, logits)
            ts.append(time.time() - t0)
        t_tok = statistics.median(ts[warmup:])
        log(f"cpu[{kind}] threads={nt}: decode at n_past=512: {t_tok * 1e3:.1f} ms/token")
        if best is None or t_tok < best[0]:
            best = (t_tok, nt)
        if time.time() - t_start > budget_s:
            break
    out.update(value=1.0 / best[0], cores=best[1], ms_per_step=best[0] * 1e3,
               sample=f"full {n_layer}-layer LLaMA-7B Q4_0, single-token evaluates at n_past=512, median of {steps} steps after {warmup} warm-up, best of the thread counts {cands}; host has {nproc} logical cores")
    m.close()
    return out


def cuda_reference(args, steps, warmup, log):
    """Prior art on the same box: the reference's own CUDA backend -- LC/ggml-cuda.cu compiled UNMODIFIED for sm_100 with cuBLAS (oracle/Makefile `refcuda`),
    driven by the reference's ggml graph executor through the LLaMA graph exactly as llm-base does with ModelParameters::use_gpu (all layers offloaded):
    dequantize + cuBLAS for batches (LC/ggml-cuda.cu:3121-3160), mul_mat_vec_q / dp4a for single tokens (:1807-1843).  Timed on the host clock around
    evaluate (the executor synchronises per node).  Checker-side code; nothing of it is linked into the product."""
    from oracle import bindings as B
    from oracle import synth
    if not B.have_ref("refcuda"):
        return {"impl": "reference-cuda", "unavailable": "oracle/_ref/libggml_refcuda.so not built (make -C oracle refcuda needs /root/reference and nvcc)"}
    hp = dict(synth.CONFIGS["7b"], n_layer=args.layers, n_ctx=N_PAST + 64, wtype=B.Q4_0)
    hp, weights = synth.make_llama_random_blocks(hp, B.Q4_0)
    ref = B.RefLib("refcuda")
    toks = synth.make_tokens(hp, N_PAST + 1)
    best = None
    for nt in (1, 4, 8):
        m = ref.llama(hp, weights, use_gpu=1, n_threads=nt, n_batch=N_PAST)
        m.eval(toks[:N_PAST])                                          # warm-up (cuBLAS handles, pools)
        pf = []
        for _ in range(3):
            m.set_n_past(0)
            t0 = time.time(); m.eval(toks[:N_PAST]); pf.append(time.time() - t0)
        logits = np.empty((1, hp["n_vocab"]), np.float32)
        ts = []
        for i in range(warmup + steps):
            m.set_n_past(N_PAST)
            t0 = time.time(); m.eval_into(toks[N_PAST:N_PAST + 1], logits); ts.append(time.time() - t0)
        t_tok, t_pf = statistics.median(ts[warmup:]), min(pf)
        log(f"reference CUDA backend, {nt} host thread(s): decode {t_tok * 1e3:.2f} ms/token ({1 / t_tok:.0f} tok/s), prefill@512 {t_pf * 1e3:.1f} ms ({N_PAST / t_pf:.0f} tok/s)")
        if best is None or t_tok < best[0]:
            best = (t_tok, t_pf, nt)
        m.close()
    prefill_metric = args.metric == "prefill"
    val = N_PAST / best[1] if prefill_metric else 1.0 / best[0]
    return {"impl": "reference-cuda", "metric": METRIC_PREFILL if prefill_metric else METRIC, "value": val, "unit": "tokens/s", "n_gpus": 1, "steps": steps, "warmup": warmup,
            "ms_per_step": (best[1] if prefill_metric else best[0]) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "reference CUDA kernels: dp4a mat-vec on Q8_1 activations (decode), dequantize -> cuBLAS (prefill)", "data": "synthetic",
            "config": {"workload": "LLaMA-7B Q4_0, the reference's own CUDA backend (LC/ggml-cuda.cu recompiled for sm_100) under its ggml graph executor", "n_layer": args.layers,
                       "host_threads": best[2]},
            "decode_tokens_per_s": 1.0 / best[0], "prefill_tokens_per_s": N_PAST / best[1], "prefill_ms": best[1] * 1e3,
            "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 4 * (N_PAST if prefill_metric else 1), "d2h_bytes_per_step": 4 * hp["n_vocab"] * (N_PAST if prefill_metric else 1)},
            "note": "not bit-exact with the reference's CPU path (its own CUDA kernels use a different summation order); context for the product's numbers, not a parity target"}


MODELS = {"7b-q4_0": dict(HP_7B), "13b-q5_1": dict(n_vocab=32000, n_embd=5120, n_head=40, n_head_kv=40, n_layer=40, n_rot=128, n_ff=13824, wtype=7)}
BLK_BYTES = {2: 18, 3: 20, 6: 22, 7: 24, 8: 34}


def dump_outputs(d, **arrays):
    """--dump-outputs: the arrays a caller of the timed path received in its last step, as float32 .npy files.  The model and the prompt are
    seeded, so two builds run with the same arguments can be compared output for output."""
    os.makedirs(d, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, np.float32))


def tp_main(args, rank, local_rank, world, steps, warmup, emit, log):
    """decode@1 at n_past = 512 of ONE model sharded by output rows over the N GPUs (strong scaling): every rank streams 1/N of the weights and its
    heads' KV cache; activation slices cross NVLink as peer stores issued by the producing kernels' epilogues as tagged 8-byte units {payload, tag} the consumers poll locally
    (llm_b200/csrc/tp.cuh) -- torch.distributed (NCCL) only brackets the timed region and takes the max over ranks."""
    import llm_b200
    from llm_b200 import _lib, tp
    from llm_b200.session import llama_tensor_shapes
    L = _lib.lib()
    hp = dict(MODELS[args.model])
    if args.layers != 32:
        hp["n_layer"] = args.layers
    name = "LLaMA-7B Q4_0" if args.model == "7b-q4_0" else "LLaMA-13B Q5_1"
    if world > 1:
        rank, local_rank, world, dist = tp.init_distributed()
    else:
        dist = None
    t0 = time.time()
    # identical weights on every rank: synthesize the FULL model on this rank's GPU (same seed), cut this rank's rows, drop the full model
    full = llm_b200.Llama(hp, llm_b200.ModelParameters(context_size=2048), device=local_rank)
    full.synthesize(0x5EED0000)
    if world > 1:
        model = tp.TpLlama(hp, llm_b200.ModelParameters(context_size=2048), None, rank=rank, world=world, device=local_rank)
        shapes = llama_tensor_shapes(hp)
        for k in shapes:
            v = full.read_tensor(k)
            rows = tp.shard_rows(k, hp, rank, world)
            if v.dtype == np.uint8:
                v = v.reshape(shapes[k][0], -1)
            model.load_tensor(k, v if rows is None else np.ascontiguousarray(v[rows[0]:rows[1]]))
        full.close()
        sess = model.start_session(llm_b200.InferenceSessionConfig(n_batch=8), dist)
    else:
        model = full
        sess = model.start_session(llm_b200.InferenceSessionConfig(n_batch=512))
    log(f"{name}: shard {rank}/{world} ready in {time.time() - t0:.1f}s; weight bytes streamed per token on this rank = {model.weight_bytes}")
    prompt = np.random.default_rng(0x70CE11).integers(0, hp["n_vocab"], N_PAST + 1, dtype=np.int32)

    def barrier():
        if dist is not None:
            import torch
            dist.barrier(device_ids=[local_rank])
            torch.cuda.synchronize()
        sess.sync()

    def allmax(*vals):
        if dist is None:
            return vals
        import torch
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return tuple(float(v) for v in t)

    t0 = time.time()
    if world > 1:                                                 # the tensor-parallel session has the decode schedule only: feed the prompt token by token
        for i in range(N_PAST):
            assert L.b200_session_evaluate(sess._s, prompt[i:i + 1].ctypes.data, 1, None, 0) == 0
    else:
        tok = np.ascontiguousarray(prompt[:N_PAST])
        assert L.b200_session_evaluate(sess._s, tok.ctypes.data, N_PAST, None, 0) == 0
    sess.sync()
    log(f"KV cache filled to n_past={N_PAST} in {time.time() - t0:.1f}s")
    one = np.ascontiguousarray(prompt[N_PAST:N_PAST + 1])
    logits = np.empty(hp["n_vocab"], np.float32)
    assert L.b200_session_evaluate(sess._s, one.ctypes.data, 1, logits.ctypes.data, 0) == 0
    launches_per_step = sess.last_launches

    def timed(n):
        for _ in range(warmup):
            sess.rewind(N_PAST); assert L.b200_session_evaluate_device(sess._s, None, 1) == 0
        barrier()
        L.b200_timing_begin()
        for _ in range(n):
            sess.rewind(N_PAST); L.b200_session_evaluate_device(sess._s, None, 1)
        ms = L.b200_timing_end_ms()
        barrier()
        return ms

    with ClockSampler(local_rank) as clk:
        ms_dev = timed(steps)
        for _ in range(3):
            sess.rewind(N_PAST); L.b200_session_evaluate(sess._s, one.ctypes.data, 1, logits.ctypes.data, 0)
        barrier()
        t0 = time.perf_counter()
        L.b200_timing_begin()
        for _ in range(steps):
            sess.rewind(N_PAST); L.b200_session_evaluate(sess._s, one.ctypes.data, 1, logits.ctypes.data, 0)
        ms_e2e = max(L.b200_timing_end_ms(), (time.perf_counter() - t0) * 1e3)
        barrier()

        def burst():
            for _ in range(32):
                sess.rewind(N_PAST); L.b200_session_evaluate_device(sess._s, None, 1)
            sess.sync()
        clk.hold(burst, agree=(lambda v: allmax(v)[0]) if world > 1 else None)
    clocks = clk.summary()
    assert np.isfinite(logits).all()
    ms_nowait = ms_local = None
    if world > 1:                                                 # the same schedule without the flag waits: what the exchange costs beyond compute + stores
        assert L.b200_session_tp_set_nowait(sess._s, 1) == 0
        ms_nowait = timed(steps)
        assert L.b200_session_tp_set_nowait(sess._s, 2) == 0       # ... and with every store kept local: compute alone
        ms_local = timed(steps)
        assert L.b200_session_tp_set_nowait(sess._s, 0) == 0
        assert sess.timeouts == 0, "a tensor-parallel flag wait timed out"
    vals = allmax(ms_dev, ms_e2e, ms_nowait if ms_nowait is not None else 0.0, ms_local if ms_local is not None else 0.0)
    ms_dev, ms_e2e = vals[0], vals[1]
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, decode_logits=logits)
    pk = peaks()
    blk = BLK_BYTES[hp["wtype"]]
    wbytes, kvbytes, embbytes = algorithmic_bytes_per_token(hp, N_PAST, blk)
    tok_bytes = wbytes + kvbytes + embbytes
    e, f = hp["n_embd"], hp["n_ff"]
    exch = hp["n_layer"] * (2 * e * 4 + (e // 32) * 64 + (f // 32) * 64) + hp["n_vocab"] * 4      # bytes every rank ends up holding per token
    line = {
        "metric": f"{name} tokens/sec (decode@1, n_past=512)" if args.model != "7b-q4_0" else METRIC,
        "value": steps / (ms_dev * 1e-3), "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8/s8 block dots -> f32", "data": "synthetic",
        "config": {"workload": f"{name} decode batch=1 n_past=512, ONE sequence on {world} GPU(s)" + (" (BASELINE.json configs[3])" if args.model == "13b-q5_1" else " (BASELINE.json configs[1])"),
                   "n_layer": hp["n_layer"], "n_ctx": 2048, "kv_cache": "f16",
                   "parallelism": (f"tp{world}: every weight matrix split by output rows (heads / n_ff / n_embd / n_vocab slices), bit-exact; activation slices are stored into every "
                                   f"peer's buffers over NVLink by the producing epilogues as tagged 8-byte units (payload + tag, one 64-bit store) that the consumers poll locally; no collective, fence or flag on the data path") if world > 1 else "single GPU",
                   "l2": "inputs larger than L2: weights streamed from HBM every step",
                   "weights": "random-init, generated on device, identical on every rank (same seed), each rank keeps its rows"},
        "e2e": {"value": steps / (ms_e2e * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": 4 * world, "d2h_bytes_per_step": 4 * hp["n_vocab"] * world, "ms_per_step": ms_e2e / steps},
        "gpu_launches": launches_per_step * steps * world, "launches_per_step": launches_per_step,
        "roofline": None,
        "step_roofline": {"bound": "hbm", "bytes_per_token": tok_bytes, "bytes_per_token_per_gpu": tok_bytes / world, "achieved_gbs": tok_bytes / (ms_dev / steps * 1e-3) / 1e9,
                          "peak": pk["hbm_gbs"] * world, "frac": tok_bytes / (ms_dev / steps * 1e-3) / 1e9 / (pk["hbm_gbs"] * world), "unit": "GB/s (all GPUs)"},
        "clocks": clocks,
        "conformance": "row split keeps every dst element one complete vec_dot: logits bit-identical to the CPU oracle (tests/test_gpu_tp.py)",
    }
    if world > 1:
        line["exchange"] = {"per_token": 4 * hp["n_layer"] + 1, "gathered_bytes_per_token_per_gpu": exch, "nvlink_bytes_per_token_per_gpu_sent": exch * (world - 1) // world,
                            "ms_per_step_without_tag_waits": vals[2] / steps, "ms_per_step_local_stores_only": vals[3] / steps,
                            "exposed_wait_share_of_step": max(0.0, 1.0 - vals[2] / ms_dev), "peer_store_share_of_step": max(0.0, (vals[2] - vals[3]) / ms_dev),
                            "relaxed_grid_waits": int(os.environ.get("B200_TP_RELAX", "0")),
                            "note": "same schedule with the tag waits skipped (garbage results) = compute + peer stores, and with every store kept local = compute alone; "
                                    "the differences are what waiting for the slowest rank's slices and what the NVLink stores cost"}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-cuda"],
                    help="reference = the reference's ggml CPU path; reference-cuda = the reference's own CUDA backend (LC/ggml-cuda.cu recompiled for sm_100, oracle/_ref) on this GPU")
    ap.add_argument("--metric", default="decode", choices=["decode", "prefill"], help="which half of BASELINE.json's metric the JSON line reports")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--layers", type=int, default=32, help="debug only: anything but 32 is NOT the benchmark config")
    ap.add_argument("--parallel", default="tp", choices=["tp", "replicas"], help="N > 1: tensor-parallel row split of ONE model (strong scaling, default) or N independent replicas")
    ap.add_argument("--model", default="7b-q4_0", choices=["7b-q4_0", "13b-q5_1"], help="13b-q5_1 = BASELINE.json configs[3] (tensor-parallel decode only)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="our arm: after the timed steps, write the logits of the last timed step (prefill: the last "
                    "row of the 512-token evaluate; decode: the token at n_past=512) as DIR/prefill_last_row_logits.npy, DIR/decode_logits.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly ONE line (the JSON); libraries that print to fd 1 (e.g. NCCL's version banner) are sent to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + "\n").encode())
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    prefill_metric = args.metric == "prefill"
    steps = args.steps if args.steps is not None else (10 if prefill_metric else 64)
    warmup = max(3, args.warmup if args.warmup is not None else (3 if prefill_metric else 8))
    metric_name = METRIC_PREFILL if prefill_metric else METRIC
    workload = ("LLaMA-7B Q4_0 prefill batch=512 from an empty session (BASELINE.json configs[2])" if prefill_metric
                else "LLaMA-7B Q4_0 decode batch=1 n_past=512 (BASELINE.json configs[1])")
    log = (lambda *a: print(*a, file=sys.stderr, flush=True)) if rank == 0 else (lambda *a: None)

    if args.impl == "reference-cuda":
        if rank == 0:
            emit(cuda_reference(args, steps, warmup, log))
        return
    if args.impl == "reference":
        if rank != 0:
            return
        rsteps, rwarm = (1, 0) if prefill_metric else (min(steps, 12), min(warmup, 3))
        cb = cpu_reference(args.metric, rsteps, rwarm, log=log, n_layer=args.layers)
        line = {"impl": "reference", "metric": metric_name, "value": cb["value"], "unit": "tokens/s", "n_gpus": args.gpus, "steps": rsteps,
                "warmup": rwarm, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "int8xint8->f32 (Q4_0 x Q8_0 blocks)", "data": "synthetic",
                "config": {"workload": workload + ", reference ggml CPU path", "n_layer": args.layers, "l2": "n/a (CPU)"},
                "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")},
                "e2e": {"value": cb["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        if "prefill_ms" in cb:
            line["prefill_ms"] = cb["prefill_ms"]
        emit(line)
        return

    # ---- our arm ----------------------------------------------------------------------------------------------------
    if (world > 1 and args.parallel == "tp") or args.model != "7b-q4_0":
        return tp_main(args, rank, local_rank, world, steps, warmup, emit, log)
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import llm_b200
    from llm_b200 import _lib
    L = _lib.lib()
    hp = dict(HP_7B, n_layer=args.layers)
    t0 = time.time()
    model = llm_b200.Llama(hp, llm_b200.ModelParameters(context_size=2048), device=local_rank)
    model.synthesize(0x5EED0000 + rank)
    log(f"model synthesized on device in {time.time() - t0:.1f}s; weight bytes streamed per token = {model.weight_bytes}")
    sess = model.start_session(llm_b200.InferenceSessionConfig(n_batch=512))
    rng = np.random.default_rng(0x70CE11 + rank)
    prompt = rng.integers(0, hp["n_vocab"], N_PAST + 1, dtype=np.int32)
    pk = peaks()

    def barrier():
        if dist is not None:
            import torch
            dist.barrier(device_ids=[local_rank])
            torch.cuda.synchronize()
        sess.sync()

    def allmax(*vals):
        if dist is None:
            return vals
        import torch
        t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return tuple(float(v) for v in t)

    # ---- prefill@512 (also fills the KV cache for the decode steps) -------------------------------------------------------------------
    tok512 = np.ascontiguousarray(prompt[:N_PAST])
    last_row = np.empty(hp["n_vocab"], np.float32)
    p_steps, p_warm = (steps, warmup) if prefill_metric else (4, 2)
    for _ in range(p_warm):                                           # the first call uploads the tokens; they stay in HBM for the device-resident arm
        sess.rewind(0)
        assert L.b200_session_evaluate(sess._s, tok512.ctypes.data, N_PAST, None, 0) == 0
    pf_launches = sess.last_launches
    barrier()
    with ClockSampler(local_rank) as pclk:
        L.b200_timing_begin()
        for _ in range(p_steps):                                      # device-resident: token ids and logits stay in HBM
            sess.rewind(0)
            L.b200_session_evaluate_device(sess._s, None, N_PAST)
        pf_dev = L.b200_timing_end_ms()
        barrier()
        t0 = time.perf_counter()
        L.b200_timing_begin()
        for _ in range(p_steps):                                      # e2e: host token ids in (2 KB), last-row logits out (128 KB), sync, every step
            sess.rewind(0)
            L.b200_session_evaluate(sess._s, tok512.ctypes.data, N_PAST, last_row.ctypes.data, 0)
        pf_e2e = max(L.b200_timing_end_ms(), (time.perf_counter() - t0) * 1e3)
        barrier()

        def pburst():
            sess.rewind(0); L.b200_session_evaluate_device(sess._s, None, N_PAST); sess.sync()
        pclk.hold(pburst)
    pf_clocks = pclk.summary()
    pf_dev, pf_e2e = allmax(pf_dev, pf_e2e)
    fl = prefill_flops(hp, N_PAST)
    pf_ms = pf_dev / p_steps
    # kernel-only timing of the weight GEMMs of one pass (the dominant kernel), on synthetic operands of the same shapes
    gemm = None
    if rank == 0:
        L.b200_op_bench_mul_mat.argtypes = [C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_float)]
        impl = 7 if os.environ.get("B200_PREFILL_GEMM", "tc5") != "mma" else 6
        e, f, v = hp["n_embd"], hp["n_ff"], hp["n_vocab"]
        tot_ms, tot_fl, n_l = 0.0, 0.0, 0
        for K, N, cnt, B in ((e, 3 * e, hp["n_layer"], N_PAST), (e, e, hp["n_layer"], N_PAST), (e, 2 * f, hp["n_layer"], N_PAST), (f, e, hp["n_layer"], N_PAST)):
            if cnt == 0:
                continue
            ms = C.c_float()
            assert L.b200_op_bench_mul_mat(hp["wtype"], K, N, B, impl, 5, C.byref(ms)) == 0
            tot_ms += ms.value * cnt; tot_fl += 2.0 * B * N * K * cnt; n_l += cnt
        gemm = dict(ms=tot_ms, flops=tot_fl, launches=n_l, impl=impl)
    prefill = {"value": world * N_PAST / (pf_ms * 1e-3), "unit": "tokens/s", "ms": pf_ms, "steps": p_steps, "launches": pf_launches,
               "e2e": {"value": world * N_PAST / (pf_e2e / p_steps * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": 4 * N_PAST, "d2h_bytes_per_step": 4 * hp["n_vocab"],
                       "ms_per_step": pf_e2e / p_steps},
               "step_roofline": {"bound": "tensor", "flops_per_step": fl, "achieved": fl / (pf_ms * 1e-3) / 1e12, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                                 "frac": fl / (pf_ms * 1e-3) / 1e12 / pk["bf16_sustained"], "peak_source": pk["source"] + " (cuBLAS bf16, sustained)"},
               "clocks": pf_clocks,
               "note": "conformant (bit-exact) path; includes attention; lm_head on the last row only (OutputRequest without all_logits) -- the reference computes all 512 rows"}
    if gemm:
        # exact-order floor: 9 fp32 operations per (token, row, 32-block) -- the reference's own rounding sequence -- on 148 SMs x 128 lanes
        fp32_floor_ms = 9.0 * gemm["flops"] / 64.0 / (148 * 128 * (pf_clocks.get("sm_mhz") or 1965.0) * 1e6) * 1e3
        prefill["roofline"] = {"bound": "tensor", "kernel": ("mm_exact_tc5_kernel<Q4_0> (tcgen05.mma + TMEM + TMA)" if gemm["impl"] == 7 else "mm_exact_mma_kernel<Q4_0> (mma.sync)") +
                               f": the {gemm['launches']} per-layer weight GEMMs of one 512-token pass, timed alone on operands of the same shapes",
                               "achieved": gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12, "peak": pk["bf16_sustained"], "unit": "TFLOP/s",
                               "frac": gemm["flops"] / (gemm["ms"] * 1e-3) / 1e12 / pk["bf16_sustained"], "peak_source": pk["source"] + " (cuBLAS bf16, sustained)",
                               "traffic": None, "launches": gemm["launches"], "ms_per_pass": gemm["ms"], "share_of_step": gemm["ms"] / pf_ms,
                               "exact_order_fp32_floor_ms": fp32_floor_ms, "frac_of_exact_order_floor": fp32_floor_ms / gemm["ms"],
                               "note": "useful flops 2*B*N*K; the bit-exact kernel runs block-diagonal MMAs (4x the useful tensor work) and is bound by the reference's ordered fp32 chain, not the tensor pipe"}
    log(f"prefill@512: {pf_ms:.2f} ms device-resident ({prefill['value']:.0f} tok/s), e2e {pf_e2e / p_steps:.2f} ms, {pf_launches} kernels" +
        (f"; weight GEMMs alone {gemm['ms']:.1f} ms" if gemm else ""))

    # ---- decode@1 at n_past = 512 -------------------------------------------------------------------------------------------------------
    d_steps, d_warm = (steps, warmup) if not prefill_metric else (16, 4)
    one = np.ascontiguousarray(prompt[N_PAST:N_PAST + 1])
    sess.rewind(0)
    assert L.b200_session_evaluate(sess._s, tok512.ctypes.data, N_PAST, None, 0) == 0      # KV cache of positions 0..511
    assert L.b200_session_evaluate(sess._s, one.ctypes.data, 1, None, 0) == 0              # leaves the token id in HBM
    launches_per_step = sess.last_launches
    for _ in range(d_warm):
        sess.rewind(N_PAST)
        assert L.b200_session_evaluate_device(sess._s, None, 1) == 0
    barrier()
    with ClockSampler(local_rank) as clk:
        L.b200_timing_begin()
        for _ in range(d_steps):
            sess.rewind(N_PAST)
            L.b200_session_evaluate_device(sess._s, None, 1)
        ms_dev = L.b200_timing_end_ms()
        barrier()
        # e2e arm: host token in, host logits out, every step
        logits = np.empty(hp["n_vocab"], np.float32)
        for _ in range(3):
            sess.rewind(N_PAST)
            L.b200_session_evaluate(sess._s, one.ctypes.data, 1, logits.ctypes.data, 0)
        barrier()
        t0 = time.perf_counter()
        L.b200_timing_begin()
        for _ in range(d_steps):
            sess.rewind(N_PAST)
            L.b200_session_evaluate(sess._s, one.ctypes.data, 1, logits.ctypes.data, 0)
        ms_e2e = L.b200_timing_end_ms()
        wall_e2e = (time.perf_counter() - t0) * 1e3
        ms_e2e = max(ms_e2e, wall_e2e)             # the host-visible time is what a caller experiences
        barrier()
        # roofline probe of the dominant kernel (quantized mat-vec) on the real weights
        nl, nbytes = C.c_int64(0), C.c_double(0)
        ms_probe = L.b200_session_probe_matvec(sess._s, 3, C.byref(nl), C.byref(nbytes))

        def burst():
            for _ in range(32):
                sess.rewind(N_PAST); L.b200_session_evaluate_device(sess._s, None, 1)
            sess.sync()
        clk.hold(burst)
    clocks = clk.summary()
    assert np.isfinite(logits).all()
    ms_dev, ms_e2e = allmax(ms_dev, ms_e2e)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, prefill_last_row_logits=last_row, decode_logits=logits)

    wbytes, kvbytes, embbytes = algorithmic_bytes_per_token(hp, N_PAST)
    tok_bytes = wbytes + kvbytes + embbytes
    probe_gbs = nbytes.value / (ms_probe * 1e-3) / 1e9
    decode = {
        "value": world * d_steps / (ms_dev * 1e-3), "unit": "tokens/s", "ms": ms_dev / d_steps, "steps": d_steps, "launches_per_step": launches_per_step,
        "e2e": {"value": world * d_steps / (ms_e2e * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": 4, "d2h_bytes_per_step": 4 * hp["n_vocab"], "ms_per_step": ms_e2e / d_steps},
        "roofline": {"bound": "hbm", "kernel": "mmv_exact_stream_kernel<Q4_0> (the stand-alone form of the mmv_fused_kernel<Q4_0,EPI> instances of the decode graph: same core loop, "
                                             "no fused epilogue): all 129 weight mat-vecs of the model back to back, timed alone (93% of a token's bytes)",
                     "achieved": probe_gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": probe_gbs / pk["hbm_gbs"], "peak_source": pk["source"] + " (burst copy)",
                     # ncu --set full (profiles/r01h_mmv_fused.ncu-rep): dram__bytes_read of a mat-vec launch = 1.0015 x its algorithmic bytes, no writes to speak of
                     "traffic": nbytes.value / max(1, nl.value) * 1.0015, "traffic_source": "ncu dram__bytes_read+write per launch, scaled from the captured w13 launch (50.80 MB vs 50.72 MB algorithmic)",
                     "launches": int(nl.value), "avg_launch_us": ms_probe * 1e3 / max(1, nl.value),
                     "algorithmic_bytes_per_launch": nbytes.value / max(1, nl.value)},
        "step_roofline": {"bound": "hbm", "bytes_per_token": tok_bytes, "weights": wbytes, "kv": kvbytes, "achieved_gbs": tok_bytes / (ms_dev / d_steps * 1e-3) / 1e9,
                          "frac": tok_bytes / (ms_dev / d_steps * 1e-3) / 1e9 / pk["hbm_gbs"]},
        "clocks": clocks,
    }
    log(f"decode@1 n_past=512: {decode['ms']:.3f} ms/token device-resident ({decode['value']:.0f} tok/s), e2e {ms_e2e / d_steps:.3f} ms; {launches_per_step} kernels per token")
    main_part, other_key, other = (prefill, "decode", decode) if prefill_metric else (decode, "prefill", prefill)
    line = {
        "metric": metric_name, "value": main_part["value"], "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": main_part["ms"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8/s8 block dots -> f32 (Q4_0 weights x Q8_0 activations)", "data": "synthetic",
        "config": {"workload": workload, "n_layer": hp["n_layer"], "n_ctx": 2048,
                   "kv_cache": "f16", "parallelism": f"{world} independent replica(s), no collective",
                   "l2": "inputs larger than L2: 3.7 GB of weights streamed per step vs 126 MB L2",
                   "weights": "random-init, generated on device (N(0,1/K) -> Q4_0 by the reference's quantizer rule)"},
        "e2e": main_part["e2e"],
        "gpu_launches": (pf_launches if prefill_metric else launches_per_step) * steps,
        "launches_per_step": pf_launches if prefill_metric else launches_per_step,
        "roofline": main_part.get("roofline"), "step_roofline": main_part["step_roofline"], "clocks": main_part["clocks"],
        other_key: other,
        "conformance": "kernels reproduce the reference's AVX2 operation order: logits and KV cache bit-identical to the reference ggml CPU path "
                       "(tests/test_gpu_llama.py::test_published_config_prefill512_and_decode_at_512; cpu_baseline.parity below for this very run)",
    }
    if not args.no_cpu_baseline and world == 1:
        try:
            # the SAME model on the CPU: device-synthesised weights read back in GGML layout, the session's KV cache installed, one step compared
            from llm_b200.session import llama_tensor_shapes
            t0 = time.time()
            weights = {}
            for k, shp in llama_tensor_shapes(hp).items():
                v = model.read_tensor(k)
                weights[k] = v.reshape(shp[0], -1) if v.dtype == np.uint8 else v
            sess.rewind(N_PAST)
            gpu_logits = np.empty(hp["n_vocab"], np.float32)
            assert L.b200_session_evaluate(sess._s, one.ctypes.data, 1, gpu_logits.ctypes.data, 0) == 0
            gpu = dict(kv=(sess.kv(0), sess.kv(1)), token=int(one[0]), logits=gpu_logits, n_past=N_PAST)
            log(f"weights + KV cache read back in {time.time() - t0:.1f}s")
            cb = cpu_reference("decode", 6, 2, log=log, weights=weights, gpu=gpu, n_layer=hp["n_layer"], budget_s=45.0)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "parity")}
            if prefill_metric:
                line["cpu_baseline"]["note"] = "decode@1 tokens/s of the reference on this host (the bounded sample); its prefill@512 is the --impl reference --metric prefill line"
        except Exception as ex:                                       # the baseline leg must never take the GPU number down
            line["cpu_baseline"] = {"value": None, "unit": "tokens/s", "cores": 0, "kind": "port", "sample": f"failed: {ex!r}"}
    emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
