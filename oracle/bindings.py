"""ctypes bindings for the oracle libraries -- TEST INFRASTRUCTURE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.

  RefLib("ref")   oracle/_ref/libggml_ref.so   the reference's own ggml.c driven by oracle/ref_harness.c
  RefLib("seam")  oracle/_ref/libggml_seam.so  the reference executor calling OUR ggml_cuda_* seam (needs a GPU)
  Oracle()        oracle/liboracle.so          the plain-C restatement (oracle/ggml_oracle.c, llama_oracle.c)
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

# enum ggml_type (LC/ggml.h:262-285)
F32, F16, Q4_0, Q4_1, Q5_0, Q5_1, Q8_0, Q8_1 = 0, 1, 2, 3, 6, 7, 8, 9
QUANT_TYPES = {"q4_0": Q4_0, "q4_1": Q4_1, "q5_0": Q5_0, "q5_1": Q5_1, "q8_0": Q8_0}
# bytes per 32-element block (LC/ggml.c:895-940)
BLOCK_BYTES = {Q4_0: 18, Q4_1: 20, Q5_0: 22, Q5_1: 24, Q8_0: 34, Q8_1: 40}
Q2_K, Q3_K, Q4_K, Q5_K, Q6_K, Q8_K = 10, 11, 12, 13, 14, 15                    # LC/ggml.h:262-285; 256-element super-blocks (LC/k_quants.h)
KQUANT_TYPES = {"q2_K": Q2_K, "q3_K": Q3_K, "q4_K": Q4_K, "q5_K": Q5_K, "q6_K": Q6_K}
SUPER_BLOCK_BYTES = {Q2_K: 84, Q3_K: 110, Q4_K: 144, Q5_K: 176, Q6_K: 210, Q8_K: 292}
VEC_DOT_TYPE = {Q4_0: Q8_0, Q4_1: Q8_1, Q5_0: Q8_0, Q5_1: Q8_1, Q8_0: Q8_0}  # LC/ggml.c:1645-1737


def row_bytes(t, k):
    if t == F32:
        return 4 * k
    if t == F16:
        return 2 * k
    if t in SUPER_BLOCK_BYTES:
        return (k // 256) * SUPER_BLOCK_BYTES[t]
    return (k // 32) * BLOCK_BYTES[t]


class RhParams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_vocab", "n_embd", "n_head", "n_head_kv", "n_layer", "n_ff", "n_rot", "n_ctx",
        "wtype", "use_gpu", "n_threads", "n_batch")]


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def have_ref(kind="ref"):
    return os.path.exists(os.path.join(HERE, "_ref", f"libggml_{kind}.so"))


class RefLib:
    """The reference ggml (unmodified) + harness."""

    def __init__(self, kind="ref"):
        path = os.path.join(HERE, "_ref", f"libggml_{kind}.so")
        self.lib = L = C.CDLL(path)
        L.rh_llama_new.restype = C.c_void_p
        L.rh_llama_new.argtypes = [C.POINTER(RhParams)]
        L.rh_llama_tensor.restype = C.c_void_p
        L.rh_llama_tensor.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_size_t)]
        L.rh_llama_finalize.argtypes = [C.c_void_p]
        L.rh_llama_reset.argtypes = [C.c_void_p]
        for fn, at in (("rh_llama_set_n_past", [C.c_void_p, C.c_int]), ("rh_llama_set_threads", [C.c_void_p, C.c_int]),
                       ("rh_llama_set_rope", [C.c_void_p, C.c_float, C.c_float])):
            if hasattr(L, fn):                                          # a prebuilt oracle/_ref of an older recipe lacks them
                getattr(L, fn).argtypes = at
        L.rh_llama_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.rh_llama_free.argtypes = [C.c_void_p]
        L.rh_llama_kv.restype = C.c_void_p
        L.rh_llama_kv.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]
        L.rh_quantize.restype = C.c_size_t
        L.rh_quantize.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int]
        L.rh_from_float.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.rh_to_float.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        L.rh_vec_dot.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.rh_fp32_to_fp16.restype = C.c_uint16
        L.rh_fp32_to_fp16.argtypes = [C.c_float]
        L.rh_fp16_to_fp32.restype = C.c_float
        L.rh_fp16_to_fp32.argtypes = [C.c_uint16]
        if hasattr(L, "rh_gpt2_new"):                                   # oracle/ref_gpt2.c
            L.rh_gpt2_new.restype = C.c_void_p
            L.rh_gpt2_new.argtypes = [C.POINTER(RgParams)]
            L.rh_gpt2_tensor.restype = C.c_void_p
            L.rh_gpt2_tensor.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_size_t)]
            L.rh_gpt2_finalize.argtypes = [C.c_void_p]
            L.rh_gpt2_reset.argtypes = [C.c_void_p]
            L.rh_gpt2_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
            L.rh_neox_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
            L.rh_gpt2_free.argtypes = [C.c_void_p]
        L.rh_op.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                            C.c_void_p, C.c_void_p, C.c_int]

    # ---- row kernels -------------------------------------------------------------------------
    def quantize(self, t, w):
        """ggml_quantize_<t> (LC/ggml.c:18083-18230) of an [N, K] f32 matrix -> uint8 [N, K/32*blk]."""
        w = np.ascontiguousarray(w, np.float32)
        n, k = w.shape
        out = np.empty((n, row_bytes(t, k)), np.uint8)
        self.lib.rh_quantize(t, _p(w), _p(out), n * k, k)
        return out

    def from_float(self, t, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty(row_bytes(t, x.size), np.uint8)
        self.lib.rh_from_float(t, _p(x), _p(out), x.size)
        return out

    def to_float(self, t, q, k):
        q = np.ascontiguousarray(q, np.uint8)
        out = np.empty(k, np.float32)
        self.lib.rh_to_float(t, _p(q), _p(out), k)
        return out

    def vec_dot(self, t, k, xq, yq):
        s = np.zeros(1, np.float32)
        self.lib.rh_vec_dot(t, k, _p(s), _p(np.ascontiguousarray(xq)), _p(np.ascontiguousarray(yq)))
        return s[0]

    def op(self, op, t, a, b, ne, iparams=(0, 0, 0, 0), fparams=(0.0, 0.0), n_threads=4, out_shape=None):
        ip = np.asarray(iparams, np.int32)
        fp = np.asarray(fparams, np.float32)
        b = np.ascontiguousarray(b)
        out = np.empty(out_shape, np.float32)
        a_p = _p(np.ascontiguousarray(a)) if a is not None else None
        rc = self.lib.rh_op(op, t, a_p, _p(b), _p(out), ne[0], ne[1], ne[2], _p(ip), _p(fp), n_threads)
        assert rc == 0, rc
        return out

    def mul_mat(self, t, wq, x, n_threads=4):
        """ggml_mul_mat(W[type; K, N], X[f32; K, B]) -> [B, N] (LC/ggml.c:10397-10586)."""
        x = np.ascontiguousarray(x, np.float32)
        b, k = x.shape
        n = wq.shape[0]
        return self.op(0, t, wq, x, (k, n, b), n_threads=n_threads, out_shape=(b, n))

    # ---- whole model ---------------------------------------------------------------------------
    def llama(self, hp, tensors, use_gpu=0, n_threads=4, n_batch=512):
        return RefLlama(self, hp, tensors, use_gpu, n_threads, n_batch)

    def gpt2(self, hp, tensors, use_gpu=0, n_threads=4, n_batch=512):
        return RefGpt2(self, hp, tensors, use_gpu, n_threads, n_batch)

    def neox(self, hp, tensors, use_gpu=0, n_threads=4, n_batch=512):
        return RefGpt2(self, hp, tensors, use_gpu, n_threads, n_batch, arch=1)


class RgParams(C.Structure):
    """rg_params (oracle/ref_gpt2.c)."""
    _fields_ = [(n, C.c_int32) for n in ("n_vocab", "n_ctx", "n_embd", "n_head", "n_layer", "wtype", "use_gpu", "n_threads", "n_batch", "has_lm_head", "arch", "n_rot", "use_parallel_residual")]


class RefGpt2:
    """The reference's GPT-2 (crates/models/gpt2) on the reference ggml: CPU build = the oracle for GPT-2, seam build = the same graph over our backend."""

    def __init__(self, ref, hp, tensors, use_gpu, n_threads, n_batch, arch=0):
        self.ref, self.hp, self.arch = ref, dict(hp), arch
        p = RgParams(arch=arch, n_rot=int(hp.get("n_rot", 0)), use_parallel_residual=int(hp.get("use_parallel_residual", 1)), **dict(**{k: int(hp[k]) for k in ("n_vocab", "n_ctx", "n_embd", "n_head", "n_layer", "wtype")}, use_gpu=use_gpu, n_threads=n_threads,
                     n_batch=n_batch, has_lm_head=int("model/lm_head" in tensors)))
        self.m = ref.lib.rh_gpt2_new(C.byref(p))
        assert self.m, "rh_gpt2_new failed"
        for name, arr in tensors.items():
            nb = C.c_size_t(0)
            dst = ref.lib.rh_gpt2_tensor(self.m, name.encode(), C.byref(nb))
            assert dst, name
            arr = np.ascontiguousarray(arr)
            assert arr.nbytes == nb.value, (name, arr.nbytes, nb.value)
            C.memmove(dst, _p(arr), arr.nbytes)
        assert ref.lib.rh_gpt2_finalize(self.m) == 0

    def eval(self, tokens):
        tokens = np.ascontiguousarray(tokens, np.int32)
        logits = np.empty((tokens.size, self.hp["n_vocab"]), np.float32)
        rc = (self.ref.lib.rh_neox_eval if self.arch else self.ref.lib.rh_gpt2_eval)(self.m, _p(tokens), tokens.size, _p(logits))
        assert rc == 0, rc
        return logits

    def close(self):
        if self.m:
            self.ref.lib.rh_gpt2_free(self.m)
            self.m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RefLlama:
    def __init__(self, ref, hp, tensors, use_gpu, n_threads, n_batch):
        self.ref, self.hp = ref, dict(hp)
        p = RhParams(**{k: int(hp[k]) for k in ("n_vocab", "n_embd", "n_head", "n_head_kv", "n_layer", "n_ff",
                                                "n_rot", "n_ctx", "wtype")},
                     use_gpu=use_gpu, n_threads=n_threads, n_batch=n_batch)
        self.m = ref.lib.rh_llama_new(C.byref(p))
        assert self.m, "rh_llama_new failed"
        for name, arr in tensors.items():
            nb = C.c_size_t(0)
            dst = ref.lib.rh_llama_tensor(self.m, name.encode(), C.byref(nb))
            assert dst, name
            arr = np.ascontiguousarray(arr)
            assert arr.nbytes == nb.value, (name, arr.nbytes, nb.value)
            C.memmove(dst, _p(arr), arr.nbytes)
        assert ref.lib.rh_llama_finalize(self.m) == 0

    def reset(self):
        self.ref.lib.rh_llama_reset(self.m)

    def set_n_past(self, n):
        self.ref.lib.rh_llama_set_n_past(self.m, int(n))

    def set_threads(self, n):
        self.ref.lib.rh_llama_set_threads(self.m, int(n))

    def set_rope(self, freq_base, freq_scale):
        self.ref.lib.rh_llama_set_rope(self.m, freq_base, freq_scale)

    def kv_ptr(self, which):
        """(address, nbytes) of the f16 K (0) / V (1) cache: lets a caller install cache contents (bench.py's CPU arm)"""
        nb = C.c_size_t(0)
        p = self.ref.lib.rh_llama_kv(self.m, which, C.byref(nb))
        return p, nb.value

    def eval(self, tokens):
        tokens = np.ascontiguousarray(tokens, np.int32)
        logits = np.empty((tokens.size, self.hp["n_vocab"]), np.float32)
        rc = self.ref.lib.rh_llama_eval(self.m, _p(tokens), tokens.size, _p(logits), None)
        assert rc == 0, rc
        return logits

    def eval_into(self, tokens, logits):
        """same, into a caller-owned [n, n_vocab] f32 buffer (timing loops: no allocation per step)"""
        tokens = np.ascontiguousarray(tokens, np.int32)
        rc = self.ref.lib.rh_llama_eval(self.m, _p(tokens), tokens.size, _p(logits), None)
        assert rc == 0, rc
        return logits

    def kv(self, which):
        nb = C.c_size_t(0)
        p = self.ref.lib.rh_llama_kv(self.m, which, C.byref(nb))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint16)), (nb.value // 2,)).copy()

    def close(self):
        if self.m:
            self.ref.lib.rh_llama_free(self.m)
            self.m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class OrHparams(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_vocab", "n_embd", "n_head", "n_head_kv", "n_layer", "n_ff", "n_rot", "n_ctx", "wtype")]


class Oracle:
    """The plain-C restatement (oracle/liboracle.so)."""

    def __init__(self, libname="liboracle.so"):
        self.lib = L = C.CDLL(os.path.join(HERE, libname))
        L.or_fp32_to_fp16.restype = C.c_uint16
        L.or_fp32_to_fp16.argtypes = [C.c_float]
        L.or_fp16_to_fp32.restype = C.c_float
        L.or_fp16_to_fp32.argtypes = [C.c_uint16]
        L.or_quantize_weights.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
        L.or_dequantize_row.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
        L.or_quantize_row_act.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
        L.or_vec_dot.restype = C.c_float
        L.or_vec_dot.argtypes = [C.c_int, C.c_int64, C.c_void_p, C.c_void_p]
        L.or_vec_dot_f16.restype = C.c_float
        L.or_vec_dot_f16.argtypes = [C.c_int64, C.c_void_p, C.c_void_p]
        L.or_mul_mat.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64]
        L.or_rms_norm.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_float]
        L.or_norm.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
        L.or_soft_max.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
        L.or_scale_mask_soft_max.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_float, C.c_int]
        L.or_silu.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.or_gelu.argtypes = [C.c_void_p, C.c_void_p, C.c_int64]
        L.or_rope.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float]
        for nm in ("or_table_silu", "or_table_gelu", "or_table_exp"):
            getattr(L, nm).restype = C.POINTER(C.c_uint16)
        L.or_llama_new.restype = C.c_void_p
        L.or_llama_new.argtypes = [C.POINTER(OrHparams)]
        L.or_llama_tensor.restype = C.c_void_p
        L.or_llama_tensor.argtypes = [C.c_void_p, C.c_char_p, C.POINTER(C.c_size_t)]
        L.or_llama_reset.argtypes = [C.c_void_p]
        L.or_llama_set_n_past.argtypes = [C.c_void_p, C.c_int]
        L.or_llama_set_rope.argtypes = [C.c_void_p, C.c_float, C.c_float]
        L.or_llama_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.or_llama_kv.restype = C.c_void_p
        L.or_llama_kv.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_size_t)]
        L.or_llama_free.argtypes = [C.c_void_p]
        L.or_llama_set_tap.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.or_llama_set_tap_stage.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]

    def fp32_to_fp16(self, x):
        return self.lib.or_fp32_to_fp16(float(x))

    def quantize(self, t, w):
        w = np.ascontiguousarray(w, np.float32)
        n, k = w.shape
        out = np.empty((n, row_bytes(t, k)), np.uint8)
        self.lib.or_quantize_weights(t, _p(w), _p(out), n, k)
        return out

    def to_float(self, t, q, k):
        q = np.ascontiguousarray(q, np.uint8)
        out = np.empty(k, np.float32)
        self.lib.or_dequantize_row(t, _p(q), _p(out), k)
        return out

    def from_float(self, t, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty(row_bytes(t, x.size), np.uint8)
        self.lib.or_quantize_row_act(t, _p(x), _p(out), x.size)
        return out

    def vec_dot(self, t, k, xq, yq):
        return np.float32(self.lib.or_vec_dot(t, k, _p(np.ascontiguousarray(xq)), _p(np.ascontiguousarray(yq))))

    def vec_dot_f16(self, x16, y16):
        x16 = np.ascontiguousarray(x16, np.uint16)
        y16 = np.ascontiguousarray(y16, np.uint16)
        return np.float32(self.lib.or_vec_dot_f16(x16.size, _p(x16), _p(y16)))

    def mul_mat(self, t, wq, x):
        x = np.ascontiguousarray(x, np.float32)
        b, k = x.shape
        n = wq.shape[0]
        out = np.empty((b, n), np.float32)
        self.lib.or_mul_mat(t, _p(np.ascontiguousarray(wq)), _p(x), _p(out), k, n, b)
        return out

    def _rows(self, fn, x, *extra):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(x)
        fn(_p(x), _p(out), x.shape[-1], x.size // x.shape[-1], *extra)
        return out

    def rms_norm(self, x, eps=5e-6):
        return self._rows(self.lib.or_rms_norm, x, C.c_float(eps))

    def norm(self, x):
        return self._rows(self.lib.or_norm, x)

    def soft_max(self, x):
        return self._rows(self.lib.or_soft_max, x)

    def scale_mask_soft_max(self, x, scale, n_past):
        """x: [nz, nr, nc] (ggml ne = [nc, nr, nz])."""
        x = np.array(x, np.float32, order="C")
        nz, nr, nc = x.shape
        self.lib.or_scale_mask_soft_max(_p(x), nc, nr, nz, scale, n_past)
        return x

    def silu(self, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(x)
        self.lib.or_silu(_p(x), _p(out), x.size)
        return out

    def gelu(self, x):
        x = np.ascontiguousarray(x, np.float32)
        out = np.empty_like(x)
        self.lib.or_gelu(_p(x), _p(out), x.size)
        return out

    def rope(self, x, n_past, n_dims, mode, freq_base=10000.0, freq_scale=1.0):
        """x: [ne2, ne1, ne0] (ggml ne = [ne0, ne1, ne2]); returns rotated copy."""
        x = np.array(x, np.float32, order="C")
        ne2, ne1, ne0 = x.shape
        self.lib.or_rope(_p(x), ne0, ne1, ne2, n_past, n_dims, mode, freq_base, freq_scale)
        return x

    def table(self, which):
        p = getattr(self.lib, f"or_table_{which}")()
        return np.ctypeslib.as_array(p, (1 << 16,)).copy()

    def llama(self, hp, tensors):
        return OracleLlama(self, hp, tensors)


class OracleLlama:
    def __init__(self, orc, hp, tensors):
        self.orc, self.hp = orc, dict(hp)
        p = OrHparams(**{k: int(hp[k]) for k in ("n_vocab", "n_embd", "n_head", "n_head_kv", "n_layer", "n_ff",
                                                 "n_rot", "n_ctx", "wtype")})
        self.m = orc.lib.or_llama_new(C.byref(p))
        for name, arr in tensors.items():
            nb = C.c_size_t(0)
            dst = orc.lib.or_llama_tensor(self.m, name.encode(), C.byref(nb))
            assert dst, name
            arr = np.ascontiguousarray(arr)
            assert arr.nbytes == nb.value, (name, arr.nbytes, nb.value)
            C.memmove(dst, _p(arr), arr.nbytes)

    def reset(self):
        self.orc.lib.or_llama_reset(self.m)

    def set_n_past(self, n):
        self.orc.lib.or_llama_set_n_past(self.m, int(n))

    def set_rope(self, freq_base, freq_scale):
        self.orc.lib.or_llama_set_rope(self.m, freq_base, freq_scale)

    def eval(self, tokens, tap_layer=None):
        tokens = np.ascontiguousarray(tokens, np.int32)
        logits = np.empty((tokens.size, self.hp["n_vocab"]), np.float32)
        tap = None
        if tap_layer is not None:
            tap = np.empty((tokens.size, self.hp["n_embd"]), np.float32)
            self.orc.lib.or_llama_set_tap(self.m, _p(tap), tap_layer)
        rc = self.orc.lib.or_llama_eval(self.m, _p(tokens), tokens.size, _p(logits))
        assert rc == 0, rc
        if tap_layer is not None:
            self.orc.lib.or_llama_set_tap(self.m, None, -2)
            return logits, tap
        return logits

    def eval_into(self, tokens, logits):
        """same as eval, into a caller-owned [n, n_vocab] f32 buffer (RefLlama's interface, used by bench.py's CPU arm)"""
        tokens = np.ascontiguousarray(tokens, np.int32)
        rc = self.orc.lib.or_llama_eval(self.m, _p(tokens), tokens.size, _p(logits))
        assert rc == 0, rc
        return logits

    def eval_tap(self, tokens, il, stage, count):
        """eval and return (logits, flat f32 tap of `count` floats taken at (layer il, stage)); see llama_oracle.c"""
        tokens = np.ascontiguousarray(tokens, np.int32)
        logits = np.empty((tokens.size, self.hp["n_vocab"]), np.float32)
        tap = np.zeros(count, np.float32)
        self.orc.lib.or_llama_set_tap_stage(self.m, _p(tap), il, stage)
        rc = self.orc.lib.or_llama_eval(self.m, _p(tokens), tokens.size, _p(logits))
        self.orc.lib.or_llama_set_tap_stage(self.m, None, -2, 11)
        assert rc == 0
        return logits, tap

    def kv_ptr(self, which):
        """(address, nbytes) of the f16 K (0) / V (1) cache, as RefLlama.kv_ptr"""
        nb = C.c_size_t(0)
        p = self.orc.lib.or_llama_kv(self.m, which, C.byref(nb))
        return p, nb.value

    def kv(self, which):
        nb = C.c_size_t(0)
        p = self.orc.lib.or_llama_kv(self.m, which, C.byref(nb))
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint16)), (nb.value // 2,)).copy()

    def close(self):
        if self.m:
            self.orc.lib.or_llama_free(self.m)
            self.m = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
