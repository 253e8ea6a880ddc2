"""CPU-side checks of the drop-in boundary: the C-ABI library loads without a GPU, exports every symbol the headers
declare, and the ggml_tensor mirror (header + ctypes) is layout-identical to the reference's struct
(LC/ggml.h:395-431; bindgen layout tests crates/ggml/sys/src/lib.rs:446).  No compute calls here."""
import ctypes as C
import json
import os
import re
import subprocess

import pytest

from conftest import GOLDEN, ROOT

LIB = os.path.join(ROOT, "llm_b200", "libllm_b200.so")


def _declared_symbols(header):
    src = open(os.path.join(ROOT, "include", header)).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b((?:ggml_(?:cuda_|init_cublas)\w*)|b200_\w+)\s*\(", src)))


def test_library_is_built():
    assert os.path.exists(LIB), "run __graft_entry__.build() first"


@pytest.mark.parametrize("header", ["ggml_b200.h", "llm_b200.h"])
def test_exports_every_declared_symbol(header):
    lib = C.CDLL(LIB)
    names = _declared_symbols(header)
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/{header} but not exported"


def test_seam_symbols_are_the_reference_bindings():
    """Every extern fn of crates/ggml/sys/src/cuda.rs:7-77 must resolve (names recorded in the golden list)."""
    rust_bound = ["ggml_init_cublas", "ggml_cuda_set_tensor_split", "ggml_cuda_mul", "ggml_cuda_can_mul_mat",
                  "ggml_cuda_mul_mat_get_wsize", "ggml_cuda_mul_mat", "ggml_cuda_host_malloc", "ggml_cuda_host_free",
                  "ggml_cuda_transform_tensor", "ggml_cuda_free_data", "ggml_cuda_assign_buffers",
                  "ggml_cuda_assign_buffers_no_scratch", "ggml_cuda_assign_buffers_force_inplace",
                  "ggml_cuda_set_main_device", "ggml_cuda_set_mul_mat_q", "ggml_cuda_set_scratch_size",
                  "ggml_cuda_free_scratch", "ggml_cuda_compute_forward"]
    lib = C.CDLL(LIB)
    for n in rust_bound:
        assert hasattr(lib, n), n
    assert sorted(rust_bound) == json.load(open(os.path.join(GOLDEN, "reference_cuda_bindings.json")))       # oracle/gen_reference_outputs.py


def test_ctypes_tensor_layout_matches_reference():
    from llm_b200 import ggml
    g = json.load(open(os.path.join(GOLDEN, "abi_layout.json")))
    T, P = ggml.Tensor, ggml.ComputeParams
    assert C.sizeof(T) == g["sizeof_tensor"] == 272
    for f in ("type", "backend", "n_dims", "ne", "nb", "op", "op_params", "is_param", "grad", "src", "perf_runs", "data", "name", "extra"):
        assert getattr(T, f).offset == g["off_" + f], f
    assert C.sizeof(P) == g["sizeof_params"]
    for f in ("type", "ith", "nth", "wsize", "wdata"):
        assert getattr(P, f).offset == g["off_p_" + f], f
    for k in ("OP_DUP", "OP_ADD", "OP_MUL", "OP_NORM", "OP_RMS_NORM", "OP_MUL_MAT", "OP_SCALE", "OP_CPY", "OP_CONT", "OP_RESHAPE",
              "OP_VIEW", "OP_PERMUTE", "OP_TRANSPOSE", "OP_GET_ROWS", "OP_DIAG_MASK_INF", "OP_SOFT_MAX", "OP_ROPE", "OP_UNARY",
              "UNARY_GELU", "UNARY_SILU"):
        assert getattr(ggml, k) == g[k], k
    assert ggml.I8 == g["TYPE_I8"] and ggml.I32 == g["TYPE_I32"] and ggml.Q8_1 == g["TYPE_Q8_1"] and ggml.TASK_COMPUTE == g["TASK_COMPUTE"]


def test_c_header_layout_matches_reference(tmp_path):
    """Compile include/ggml_b200.h with gcc and compare sizeof/offsetof/enums with the values dumped from LC/ggml.h."""
    g = json.load(open(os.path.join(GOLDEN, "abi_layout.json")))
    fields = ["type", "backend", "n_dims", "ne", "nb", "op", "op_params", "is_param", "grad", "src", "perf_runs", "data", "name", "extra"]
    prog = ['#include "ggml_b200.h"', "#include <stdio.h>", "#include <stddef.h>", "int main(void){",
            'printf("{\\"sizeof_tensor\\":%zu", sizeof(struct ggml_tensor));']
    for f in fields:
        prog.append(f'printf(",\\"off_{f}\\":%zu", offsetof(struct ggml_tensor, {f}));')
    prog.append('printf(",\\"sizeof_params\\":%zu", sizeof(struct ggml_compute_params));')
    for f in ("type", "ith", "nth", "wsize", "wdata"):
        prog.append(f'printf(",\\"off_p_{f}\\":%zu", offsetof(struct ggml_compute_params, {f}));')
    for k in ("DUP", "ADD", "MUL", "NORM", "RMS_NORM", "MUL_MAT", "SCALE", "CPY", "CONT", "RESHAPE", "VIEW", "PERMUTE", "TRANSPOSE",
              "GET_ROWS", "DIAG_MASK_INF", "SOFT_MAX", "ROPE", "UNARY"):
        prog.append(f'printf(",\\"OP_{k}\\":%d", B200_OP_{k});')
    prog.append('printf(",\\"UNARY_GELU\\":%d,\\"UNARY_SILU\\":%d,\\"TYPE_I8\\":%d,\\"TYPE_I16\\":%d,\\"TYPE_I32\\":%d,\\"TYPE_Q8_1\\":%d,\\"TASK_COMPUTE\\":%d}\\n",'
                ' B200_UNARY_GELU, B200_UNARY_SILU, B200_TYPE_I8, B200_TYPE_I16, B200_TYPE_I32, B200_TYPE_Q8_1, B200_TASK_COMPUTE);')
    prog.append("return 0;}")
    src = tmp_path / "p.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "p"
    subprocess.check_call(["/usr/bin/gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    mine = json.loads(subprocess.check_output([str(exe)]))
    assert mine == g


def test_python_package_fails_loudly_without_library(monkeypatch):
    from llm_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libllm_b200.so")
    with pytest.raises(ImportError):
        _lib.lib()
