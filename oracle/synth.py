"""Seeded synthetic LLaMA-shaped GGML models for parity tests -- TEST INFRASTRUCTURE.

Follows SURVEY.md §8(d): every 2-D weight ~ N(0, 1/K) in f32 then quantized with the reference's
ggml_quantize_<type> (the call crates/llm-base/src/quantize.rs:365-377 makes, which quantizes every
".*weight" 2-D tensor including tok_embeddings/output, crates/models/llama/src/lib.rs:390-392);
norm gains 1 + 0.1 N(0,1) kept f32. Tensor names are the loader's (llama lib.rs:52-91).
"""
import numpy as np

from . import bindings as B

CONFIGS = {
    # tiny shapes the CPU oracle finishes in milliseconds; K multiples of 64 (Q4 row rule, crates/ggml/src/lib.rs:112-118)
    "tiny":   dict(n_vocab=320, n_embd=256, n_head=4, n_head_kv=4, n_layer=2, n_ff=704, n_rot=64, n_ctx=128),
    # shapes the one-launch decode kernel accepts (K % 256 == 0), incl. grouped-query attention
    "tiny8":  dict(n_vocab=320, n_embd=256, n_head=4, n_head_kv=4, n_layer=2, n_ff=768, n_rot=64, n_ctx=128),
    "gqa8":   dict(n_vocab=352, n_embd=512, n_head=8, n_head_kv=2, n_layer=3, n_ff=1024, n_rot=64, n_ctx=256),
    "small":  dict(n_vocab=1024, n_embd=512, n_head=8, n_head_kv=8, n_layer=3, n_ff=1408, n_rot=64, n_ctx=256),
    # 7B layer geometry with few layers (BASELINE.json configs[1]/[2] shapes; SURVEY.md §8)
    "7b-2l":  dict(n_vocab=32000, n_embd=4096, n_head=32, n_head_kv=32, n_layer=2, n_ff=11008, n_rot=128, n_ctx=1024),
    "7b":     dict(n_vocab=32000, n_embd=4096, n_head=32, n_head_kv=32, n_layer=32, n_ff=11008, n_rot=128, n_ctx=2048),
    "13b":    dict(n_vocab=32000, n_embd=5120, n_head=40, n_head_kv=40, n_layer=40, n_ff=13824, n_rot=128, n_ctx=2048),
}


def tensor_shapes(hp):
    """name -> (ne1 rows N, ne0 cols K) for 2-D weights, (n,) for 1-D."""
    e, f, v = hp["n_embd"], hp["n_ff"], hp["n_vocab"]
    gqa = e // (hp["n_head"] // hp["n_head_kv"])
    shapes = {"tok_embeddings.weight": (v, e), "norm.weight": (e,), "output.weight": (v, e)}
    for i in range(hp["n_layer"]):
        p = f"layers.{i}."
        shapes[p + "attention_norm.weight"] = (e,)
        shapes[p + "attention.wq.weight"] = (e, e)
        shapes[p + "attention.wk.weight"] = (gqa, e)
        shapes[p + "attention.wv.weight"] = (gqa, e)
        shapes[p + "attention.wo.weight"] = (e, e)
        shapes[p + "ffn_norm.weight"] = (e,)
        shapes[p + "feed_forward.w1.weight"] = (f, e)
        shapes[p + "feed_forward.w2.weight"] = (e, f)
        shapes[p + "feed_forward.w3.weight"] = (f, e)
    return shapes


def make_llama(hp, wtype, quantize, seed=0x5EED0000, gain=1.0):
    """Returns (hp_with_wtype, {name: ndarray}) -- uint8 block rows for 2-D weights, f32 for norms.

    `quantize(type, f32[N,K]) -> uint8[N, row_bytes]` is the reference quantizer (RefLib.quantize) or
    its restatement (Oracle.quantize); tests assert the two agree bit for bit.
    """
    hp = dict(hp, wtype=wtype)
    out = {}
    for idx, (name, shp) in enumerate(tensor_shapes(hp).items()):
        rng = np.random.default_rng(seed + idx)
        if len(shp) == 1:
            out[name] = (1.0 + 0.1 * rng.standard_normal(shp)).astype(np.float32)
        else:
            n, k = shp
            w = (rng.standard_normal((n, k)) * (gain / np.sqrt(k))).astype(np.float32)
            out[name] = quantize(wtype, w)
    return hp, out


def make_llama_random_blocks(hp, wtype, seed=0x5EED0000):
    """A full-size model in seconds: the quantized blocks are drawn directly (uniform quants, fp16 scales ~ U[0.5, 1.5] * 2 / (15 sqrt(K)))
    instead of quantizing 7e9 gaussians -- for TIMING the reference on the published configuration (bench.py --impl reference); parity
    tests use make_llama or device-synthesised weights read back."""
    hp = dict(hp, wtype=wtype)
    rng = np.random.default_rng(seed)
    bb = B.BLOCK_BYTES[wtype]
    out = {}
    for name, shp in tensor_shapes(hp).items():
        if len(shp) == 1:
            out[name] = (1.0 + 0.1 * rng.standard_normal(shp)).astype(np.float32)
            continue
        n, k = shp
        nb = k // 32
        blk = rng.integers(0, 256, size=(n, nb, bb), dtype=np.uint8)
        d = ((rng.random((n, nb), dtype=np.float32) + 0.5) * np.float32(2.0 / (15.0 * np.sqrt(k)))).astype(np.float16)
        blk[:, :, 0:2] = d.view(np.uint8).reshape(n, nb, 2)
        if wtype in (B.Q4_1, B.Q5_1):              # {d, m}: a small finite min
            m = (-rng.random((n, nb), dtype=np.float32) / np.float32(np.sqrt(k))).astype(np.float16)
            blk[:, :, 2:4] = m.view(np.uint8).reshape(n, nb, 2)
        out[name] = blk.reshape(n, nb * bb)
    return hp, out


# byte offsets of the fp16 super-block scale d (and dmin) in block_q2_K .. block_q6_K (LC/k_quants.h)
KQUANT_FP16_FIELDS = {B.Q2_K: (80, 82), B.Q3_K: (108,), B.Q4_K: (0, 2), B.Q5_K: (0, 2), B.Q6_K: (208,)}


def make_kquant_blocks(t, n, k, seed):
    """[n, k/256 * block bytes] uint8 rows of K-quant type t drawn directly: uniform bytes for the quants and the packed sub-block scales and
    mins (every bit pattern is a valid block), fp16 d / dmin ~ U[0.5, 1.5] / 1024.  Weights for the K-quant kernel tests without the
    reference's quantizer; the expected products of these rows are recorded from the reference (oracle/gen_reference_outputs.py)."""
    rng = np.random.default_rng(seed)
    bb, nb = B.SUPER_BLOCK_BYTES[t], k // 256
    blk = rng.integers(0, 256, size=(n, nb, bb), dtype=np.uint8)
    for off in KQUANT_FP16_FIELDS[t]:
        d = ((rng.random((n, nb), dtype=np.float32) + 0.5) / np.float32(1024.0)).astype(np.float16)
        blk[:, :, off:off + 2] = d.view(np.uint8).reshape(n, nb, 2)
    return blk.reshape(n, nb * bb)


def make_tokens(hp, n, seed=0x70CE11):
    return np.random.default_rng(seed).integers(0, hp["n_vocab"], size=n, dtype=np.int32)


# ---- GPT-2 (BASELINE.json configs[0]; tensor names of crates/models/gpt2/src/lib.rs:59-107) -------------------------------------------
GPT2_CONFIGS = {
    "gpt2-tiny": dict(n_vocab=320, n_ctx=64, n_embd=128, n_head=4, n_layer=2),
    "gpt2-117m": dict(n_vocab=50257, n_ctx=1024, n_embd=768, n_head=12, n_layer=12),
}


def gpt2_tensor_shapes(hp, lm_head=False):
    e, v, c = hp["n_embd"], hp["n_vocab"], hp["n_ctx"]
    shapes = {"model/wpe": (c, e), "model/wte": (v, e), "model/ln_f/g": (e,), "model/ln_f/b": (e,)}
    if lm_head:
        shapes["model/lm_head"] = (v, e)
    for i in range(hp["n_layer"]):
        p = f"model/h{i}/"
        shapes.update({p + "ln_1/g": (e,), p + "ln_1/b": (e,), p + "ln_2/g": (e,), p + "ln_2/b": (e,),
                       p + "attn/c_attn/w": (3 * e, e), p + "attn/c_attn/b": (3 * e,), p + "attn/c_proj/w": (e, e), p + "attn/c_proj/b": (e,),
                       p + "mlp/c_fc/w": (4 * e, e), p + "mlp/c_fc/b": (4 * e,), p + "mlp/c_proj/w": (e, 4 * e), p + "mlp/c_proj/b": (e,)})
    return shapes


def make_gpt2(hp, wtype, quantize, seed=0x6F720000, lm_head=False):
    """SURVEY.md §8(d): 2-D weights N(0, 1/K) quantized with the reference quantizer (wpe stays f32), gains 1 + 0.1 N(0,1), biases 0.01 N(0,1)."""
    hp = dict(hp, wtype=wtype)
    out = {}
    for idx, (name, shp) in enumerate(gpt2_tensor_shapes(hp, lm_head).items()):
        rng = np.random.default_rng(seed + idx)
        if len(shp) == 1:
            out[name] = ((1.0 if name.endswith("/g") else 0.0) + (0.1 if name.endswith("/g") else 0.01) * rng.standard_normal(shp)).astype(np.float32)
        else:
            n, k = shp
            w = (rng.standard_normal((n, k)) / np.sqrt(k)).astype(np.float32)
            out[name] = w if name == "model/wpe" else quantize(wtype, w)
    return hp, out


# ---- GPT-NeoX (BASELINE.json configs[4] geometry; tensor names of crates/models/gptneox/src/lib.rs:58-123) ------------------------------------
NEOX_CONFIGS = {
    "neox-tiny": dict(n_vocab=384, n_ctx=64, n_embd=128, n_head=4, n_layer=2, n_rot=8, use_parallel_residual=1),
    "neox-tiny-seq": dict(n_vocab=384, n_ctx=64, n_embd=128, n_head=4, n_layer=2, n_rot=32, use_parallel_residual=0),
    "neox-20b": dict(n_vocab=50432, n_ctx=2048, n_embd=6144, n_head=64, n_layer=44, n_rot=24, use_parallel_residual=1),
}


def neox_tensor_shapes(hp):
    e, v = hp["n_embd"], hp["n_vocab"]
    shapes = {"gpt_neox.embed_in.weight": (v, e), "gpt_neox.final_layer_norm.weight": (e,), "gpt_neox.final_layer_norm.bias": (e,), "embed_out.weight": (v, e)}
    for i in range(hp["n_layer"]):
        p = f"gpt_neox.layers.{i}."
        shapes.update({p + "input_layernorm.weight": (e,), p + "input_layernorm.bias": (e,),
                       p + "post_attention_layernorm.weight": (e,), p + "post_attention_layernorm.bias": (e,),
                       p + "attention.query_key_value.weight": (3 * e, e), p + "attention.query_key_value.bias": (3 * e,),
                       p + "attention.dense.weight": (e, e), p + "attention.dense.bias": (e,),
                       p + "mlp.dense_h_to_4h.weight": (4 * e, e), p + "mlp.dense_h_to_4h.bias": (4 * e,),
                       p + "mlp.dense_4h_to_h.weight": (e, 4 * e), p + "mlp.dense_4h_to_h.bias": (e,)})
    return shapes


def make_neox(hp, wtype, quantize, seed=0x4E580000):
    hp = dict(hp, wtype=wtype)
    out = {}
    for idx, (name, shp) in enumerate(neox_tensor_shapes(hp).items()):
        rng = np.random.default_rng(seed + idx)
        if len(shp) == 1:
            gain = name.endswith("norm.weight")
            out[name] = ((1.0 if gain else 0.0) + (0.1 if gain else 0.01) * rng.standard_normal(shp)).astype(np.float32)
        else:
            n, k = shp
            out[name] = quantize(wtype, (rng.standard_normal((n, k)) / np.sqrt(k)).astype(np.float32))
    return hp, out
