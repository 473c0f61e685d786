"""GPU cross-check against the UNMODIFIED reference extension on identical tensors -- SURVEY.md 8c row (iv).  The
reference's outputs are stored in tests/golden (reference_parity.npz and the reconstruct of linear_<name>.npz, written by
oracle/gen_golden.py on a B200 with the reference extension built by oracle/build_ref.py); the inputs come from the seeded
generators of tests/cases.py.

Contract (SURVEY.md 8c tolerance row):
  reconstruct                bit-exact
  gemm (M <= 32, force_cuda) rel_l2(new, ref) <= 1e-3  and  rel_l2(new, truth) <= rel_l2(ref, truth) + 1e-5
  rms_norm                   <= 1 fp16 ulp;   rope: bit-exact;   Q4 kv pack/unpack: bit-exact (same intrinsics)
"""
import os

import numpy as np
import pytest
import torch

import cases
import exl2_oracle as oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLD, "reference_parity.npz"))


def _mine(name):
    from exllamav2_b200.linear import ExLlamaV2Linear, load_tensor_dict
    w_np = cases.make_case(name)
    K, N = cases.case_shape(name)
    lin = ExLlamaV2Linear(K, N, has_bias="bias" in w_np, device=DEV)
    lin.load(load_tensor_dict(w_np, DEV))
    return lin, w_np


# the reference's kernels need N % 32 == 0 style tiles; keep to the shapes it supports
REF_CASES = cases.ref_cases()


@pytest.mark.parametrize("name", REF_CASES)
def test_reconstruct_matches_reference(name):
    lin, w_np = _mine(name)
    W_ref = np.load(os.path.join(GOLD, f"linear_{name}.npz"))["reconstruct"]
    W_new = lin.get_weight_tensor_dq()
    assert np.array_equal(W_ref, W_new.cpu().numpy().view(np.uint16))
    lin.unload()


@pytest.mark.parametrize("name", REF_CASES)
@pytest.mark.parametrize("M", cases.REF_GEMM_M)
def test_gemm_matches_reference(ref, name, M):
    lin, w_np = _mine(name)
    a = cases.activations(name, M)
    at = torch.from_numpy(a).to(DEV)
    c_ref = ref[f"gemm_{name}_m{M}"].view(np.float16)
    c_new = lin.forward(at)
    W = oracle.exl2_reconstruct(w_np) if name in cases.EXL2_CASES else oracle.gptq_reconstruct(w_np)
    truth = oracle.gemm_truth(a, W, w_np.get("bias"))
    e_ref = oracle.rel_l2(c_ref, truth)
    e_new = oracle.rel_l2(c_new.cpu().numpy(), truth)
    e_x = oracle.rel_l2(c_new.cpu().numpy(), c_ref.astype(np.float32))
    assert e_x <= 1e-3 + e_ref, f"new vs ref {e_x:.2e} (ref vs truth {e_ref:.2e})"
    assert e_new <= e_ref + 1e-5, f"new {e_new:.2e} is further from truth than ref {e_ref:.2e}"
    lin.unload()


def test_ops_match_reference(ref):
    from exllamav2_b200 import ext as ext_c
    from exllamav2_b200.ext import none_tensor
    d = {k: torch.from_numpy(v).to(DEV) for k, v in cases.ref_ops_inputs().items()}
    # rms_norm
    y_new = torch.empty_like(d["norm_x"])
    ext_c.rms_norm(d["norm_x"], d["norm_w"], y_new, 1e-5)
    diff = np.abs(ref["norm_y"].view(np.int16).astype(np.int32) - y_new.view(torch.int16).cpu().numpy().astype(np.int32))
    assert diff.max() <= 1
    # rope (both styles), with per-batch offsets
    hd, heads = 128, 8
    sin, cos = oracle.rope_tables(hd, 128)
    st, ct = torch.from_numpy(sin).to(DEV), torch.from_numpy(cos).to(DEV)
    offs = torch.tensor([0, 11], dtype=torch.int, device=DEV)
    for tag, neox in (("neox", True), ("gptj", False)):
        b = d[f"rope_{tag}_x"].clone()
        ext_c.rope_(b, st, ct, 17, heads, hd, offs, neox)
        assert np.array_equal(ref[f"rope_{tag}_y"], b.cpu().numpy().view(np.uint16)), f"rope neox={neox}"
    # Q4 kv
    k, v = d["kv_k"], d["kv_v"]
    kq = torch.zeros((2, 9, 8, 64), dtype=torch.uint8, device=DEV)
    ks = torch.zeros((2, 9, 8, 4), dtype=torch.half, device=DEV)
    vq, vs = torch.zeros_like(kq), torch.zeros_like(ks)
    ext_c.fp16_to_q_kv(k, kq, ks, v, vq, vs, 2, 2, 6, 0, none_tensor, none_tensor, 4)
    ko, vo = torch.zeros_like(k), torch.zeros_like(v)
    ext_c.q_to_fp16_kv(kq, ko, ks, vq, vo, vs, 2, 2, 6, 0, none_tensor, none_tensor, 4)
    for key, n in (("kq", kq), ("ks", ks), ("vq", vq), ("vs", vs), ("ko", ko), ("vo", vo)):
        assert np.array_equal(ref[f"kv_{key}"], n.view(torch.uint8).cpu().numpy()), key
