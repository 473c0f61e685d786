"""The C-ABI library loads without a GPU and exports every symbol include/exl2_b200.h declares; host-only entry
points behave; the product refuses CPU tensors (no CPU fallback)."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from exllamav2_b200 import build
    return ctypes.CDLL(build.build())


def test_every_declared_symbol_is_exported(lib):
    hdr = open(os.path.join(ROOT, "include", "exl2_b200.h")).read()
    names = sorted(set(re.findall(r"\b(exl2b_[a-z0-9_]+)\s*\(", hdr)))
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported"


def test_make_group_map_matches_oracle():
    import exl2_oracle as oracle
    from exllamav2_b200 import ext as ext_c
    q_groups = np.array([8, 0, 6, 8, 5, 32, 5, 52], dtype=np.int16)      # (bits, first packed row)
    num_qrows = 72
    got = ext_c.make_group_map(torch.from_numpy(q_groups), num_qrows).numpy()
    assert np.array_equal(got, oracle.make_group_map(q_groups, num_qrows))


def test_cpu_tensors_are_rejected():
    from exllamav2_b200 import ext as ext_c
    x = torch.zeros((1, 64), dtype=torch.half)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ext_c.rms_norm(x, torch.ones(64, dtype=torch.half), x.clone(), 1e-5)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        ext_c.make_q_matrix(torch.zeros((8, 64), dtype=torch.int32), *([ext_c.none_tensor] * 11), 0)


def test_error_message_plumbing(lib):
    lib.exl2b_last_error.restype = ctypes.c_char_p
    lib.exl2b_qmatrix_info.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 5
    assert lib.exl2b_qmatrix_info(None, None, None, None, None, None) != 0
    assert b"null handle" in lib.exl2b_last_error()


def test_hot_path_names_cover_reference_call_sites():
    """Every ext_c.<name> the reference's hot-path files call for a Llama-family quantized model must exist in our
    module (SURVEY.md 8b).  The names are stored in tests/golden/reference_ext_calls.json (oracle/gen_golden.py --ext-calls)."""
    from exllamav2_b200 import ext as ext_c
    for n in ext_c.HOT_PATH_EXPORTS:
        assert callable(getattr(ext_c, n))
    with open(os.path.join(ROOT, "tests", "golden", "reference_ext_calls.json")) as f:
        used = set(json.load(f)["names"])
    assert {"gemm_half_q_half", "reconstruct", "rms_norm", "fp16_to_q_kv", "q_to_fp16_kv"} <= used
    out_of_scope = {  # other families / TP single-process glue / FP8 / load_in_q4 debug mode (SURVEY.md 2.2)
        "tensor_remap", "tensor_remap_4bit", "matrix_fp16_to_q4", "matrix_q4_to_fp16", "gemm_half_q_half_tp",
        "make_q_matrix_split", "tp_all_reduce", "fp16_to_fp8", "fp8_to_fp16", "count_match", "rms_norm_tp",
        "cache_rotate", "layer_norm", "layer_norm_", "head_norm", "head_norm_",
    }
    missing = sorted(n for n in used - out_of_scope if not hasattr(ext_c, n))
    assert not missing, f"hot-path names missing from the drop-in module: {missing}"
