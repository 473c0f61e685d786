#!/usr/bin/env python
"""Generate golden vectors by running the UNMODIFIED reference CUDA extension (oracle/_ref, built by
oracle/build_ref.py) on a GPU over the seeded cases of tests/cases.py.  TEST INFRASTRUCTURE.

    python oracle/gen_golden.py [outdir]        (default gpurun_out/golden; copy the .npz files to tests/golden/)
    python oracle/gen_golden.py --parity [outdir]      (GPU; writes reference_parity.npz, default tests/golden)
    python oracle/gen_golden.py --ext-calls [outdir]   (CPU; writes reference_ext_calls.json, default tests/golden)

The reference has no golden vectors of its own for this path (SURVEY.md 8c); these files are what pins the CPU
oracle (tests/test_oracle_golden.py) and, on the GPU box, our kernels (tests/test_gpu_golden.py).
Outputs per case:  reconstruct (fp16 bits), gemm force_cuda for several M (fp16 bits; NOT bit-reproducible across
runs because the reference accumulates with fp16 atomics), plus rms_norm / rope / Q4-kv vectors.

--parity stores the reference's outputs on the inputs of tests/test_gpu_vs_reference.py and of the GPTQ 4096 x 4096 row
of tests/test_gpu_row_blocks.py; --ext-calls stores the ext_c.<name> calls of the reference's hot-path Python files
(tests/test_abi.py).  With them the tests compare with the reference without needing its sources or binaries.
"""
import json
import os
import re
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import cases  # noqa: E402
import exl2_oracle as oracle  # noqa: E402
from build_ref import REF_ROOT, load_ref  # noqa: E402

DEV = "cuda:0"
GOLD = os.path.join(ROOT, "tests", "golden")
none_tensor = torch.empty((1, 1), device="meta")


def ref_make_q_matrix(ref, w_np, prescale=1.0, offset_qzeros=False):
    """The reference's Python glue (exllamav2/ext.py:325-410, module.py:118-121) driving the reference extension."""
    w = {k: (torch.from_numpy(np.ascontiguousarray(v)) if k == "g_idx" else torch.from_numpy(np.ascontiguousarray(v)).to(DEV))
         for k, v in w_np.items()}
    if "q_weight" in w:
        w["q_perm"] = torch.argsort(w["q_invperm"]).to(torch.int)
        w["q_scale_max"] *= prescale / 256
        w["q_perm"] = w["q_perm"].short()
        w["q_invperm"] = w["q_invperm"].short()
        gm = ref.make_group_map(w["q_groups"].cpu(), w["q_weight"].shape[0]).to(DEV)
        w["q_group_map"] = gm
        K, N = w["q_perm"].shape[0], w["q_weight"].shape[1]
        temp_dq = torch.empty((K * N,), dtype=torch.half, device=DEV)
        h = ref.make_q_matrix(w["q_weight"], w["q_perm"], w["q_invperm"], w["q_scale"], w["q_scale_max"], w["q_groups"],
                              w["q_group_map"], none_tensor, none_tensor, none_tensor, w.get("bias", none_tensor), temp_dq, K)
    else:
        if offset_qzeros:
            w["qzeros"] -= 0b00010001000100010001000100010001
        K, N = w["qweight"].shape[0] * 8, w["qweight"].shape[1]
        temp_dq = torch.empty((K * N,), dtype=torch.half, device=DEV)
        if not (w["g_idx"] == 0).all().item():
            w["q_perm"] = torch.empty((K,), dtype=torch.short, device=DEV)
            w["q_invperm"] = torch.empty_like(w["q_perm"])
            h = ref.make_q_matrix(w["qweight"], w["q_perm"], w["q_invperm"], none_tensor, none_tensor, none_tensor, none_tensor,
                                  w["qzeros"], w["scales"], w["g_idx"].cpu(), w.get("bias", none_tensor), temp_dq, K)
        else:
            h = ref.make_q_matrix(w["qweight"], none_tensor, none_tensor, none_tensor, none_tensor, none_tensor, none_tensor,
                                  w["qzeros"], w["scales"], none_tensor, w.get("bias", none_tensor), temp_dq, K)
    torch.cuda.synchronize()
    return h, w, temp_dq, (K, N)


def main(outdir):
    ref = load_ref()
    if ref is None:
        print("oracle/_ref/exllamav2_ext_ref.so not built; run oracle/build_ref.py where /root/reference exists")
        return 1
    os.makedirs(outdir, exist_ok=True)
    names = [n for n in list(cases.EXL2_CASES) + list(cases.GPTQ_CASES)]
    skipped = []
    for name in names:
        K, N = cases.case_shape(name)
        if N % 32 != 0:   # the reference kernels assume 4-column vectors / 32-column tiles for these widths
            pass
        w_np = cases.make_case(name)
        try:
            h, w, temp_dq, _ = ref_make_q_matrix(ref, w_np)
        except Exception as e:  # pragma: no cover
            skipped.append((name, repr(e)))
            continue
        out = {}
        W = torch.empty((K, N), dtype=torch.half, device=DEV)
        ref.reconstruct(h, W)
        out["reconstruct"] = W.cpu().numpy().view(np.uint16)
        for M in cases.M_VALUES:
            a = torch.from_numpy(cases.activations(name, M)).to(DEV)
            c = torch.empty((M, N), dtype=torch.half, device=DEV)
            ref.gemm_half_q_half(a, h, c, True)
            out[f"gemm_m{M}"] = c.cpu().numpy().view(np.uint16)
        torch.cuda.synchronize()
        ref.free_q_matrix(h)
        np.savez_compressed(os.path.join(outdir, f"linear_{name}.npz"), **out)
        print("golden", name, {k: v.shape for k, v in out.items()})

    # rms_norm / rope / kv
    rng = np.random.default_rng(77)
    ops = {}
    x = rng.normal(0, 1.5, size=(3, 2048)).astype(np.float16)
    w = (1 + 0.1 * rng.normal(size=(2048,))).astype(np.float16)
    y = torch.empty((3, 2048), dtype=torch.half, device=DEV)
    ref.rms_norm(torch.from_numpy(x).to(DEV), torch.from_numpy(w).to(DEV), y, 1e-5)
    ops["norm_x"], ops["norm_w"], ops["norm_y"] = x.view(np.uint16), w.view(np.uint16), y.cpu().numpy().view(np.uint16)
    hd, heads = 128, 4
    sin, cos = oracle.rope_tables(hd, 64)
    for neox in (True, False):
        xr = rng.normal(0, 1, size=(2, 3, heads * hd)).astype(np.float16)
        xt = torch.from_numpy(xr).to(DEV)
        offs = torch.tensor([0, 5], dtype=torch.int, device=DEV)
        ref.rope_(xt, torch.from_numpy(sin).to(DEV)[None, None], torch.from_numpy(cos).to(DEV)[None, None], 9, heads, hd, offs, neox)
        tag = "neox" if neox else "gptj"
        ops[f"rope_{tag}_x"], ops[f"rope_{tag}_y"] = xr.view(np.uint16), xt.cpu().numpy().view(np.uint16)
    ops["rope_sin"], ops["rope_cos"] = sin.view(np.uint16), cos.view(np.uint16)
    kv = rng.normal(0, 1, size=(2, 4, 8, 128)).astype(np.float16)
    kt = torch.from_numpy(kv).to(DEV)
    kq = torch.zeros((2, 4, 8, 64), dtype=torch.uint8, device=DEV)
    ks = torch.zeros((2, 4, 8, 4), dtype=torch.half, device=DEV)
    vq, vs = torch.zeros_like(kq), torch.zeros_like(ks)
    ref.fp16_to_q_kv(kt, kq, ks, kt, vq, vs, 2, 0, 4, 0, none_tensor, none_tensor, 4)
    ko, vo = torch.zeros_like(kt), torch.zeros_like(kt)
    ref.q_to_fp16_kv(kq, ko, ks, vq, vo, vs, 2, 0, 4, 0, none_tensor, none_tensor, 4)
    ops["kv_x"], ops["kv_q"], ops["kv_s"], ops["kv_y"] = kv.view(np.uint16), kq.cpu().numpy(), ks.cpu().numpy().view(np.uint16), ko.cpu().numpy().view(np.uint16)
    np.savez_compressed(os.path.join(outdir, "ops.npz"), **ops)
    print("golden ops", {k: v.shape for k, v in ops.items()})
    if skipped:
        print("SKIPPED:", skipped)
    return 0


def parity(outdir):
    ref = load_ref()
    if ref is None:
        print("oracle/_ref/exllamav2_ext_ref.so not built; run oracle/build_ref.py where the reference sources exist")
        return 1
    out = {}
    for name in cases.ref_cases():
        w_np = cases.make_case(name)
        h, keep, temp_dq, (K, N) = ref_make_q_matrix(ref, w_np)
        # the reconstruct comparison reads the committed linear_<name>.npz: it must still be what the reference computes
        W = torch.empty((K, N), dtype=torch.half, device=DEV)
        ref.reconstruct(h, W)
        gold = np.load(os.path.join(GOLD, f"linear_{name}.npz"))["reconstruct"]
        assert np.array_equal(W.cpu().numpy().view(np.uint16), gold), f"{name}: reconstruct differs from linear_{name}.npz"
        for M in cases.REF_GEMM_M:
            c = torch.empty((M, N), dtype=torch.half, device=DEV)
            ref.gemm_half_q_half(torch.from_numpy(cases.activations(name, M)).to(DEV), h, c, True)
            out[f"gemm_{name}_m{M}"] = c.cpu().numpy().view(np.uint16)
        ref.free_q_matrix(h)
    for act_order in (False, True):
        w_np, a = cases.gptq_4096_row(act_order)
        h, keep, temp_dq, (K, N) = ref_make_q_matrix(ref, w_np)
        c = torch.empty((1, N), dtype=torch.half, device=DEV)
        ref.gemm_half_q_half(torch.from_numpy(a).to(DEV), h, c, True)
        out[f"gptq4096_act{int(act_order)}"] = c.cpu().numpy().view(np.uint16)
        ref.free_q_matrix(h)

    d = {k: torch.from_numpy(v).to(DEV) for k, v in cases.ref_ops_inputs().items()}
    y = torch.empty_like(d["norm_x"])
    ref.rms_norm(d["norm_x"], d["norm_w"], y, 1e-5)
    out["norm_y"] = y.cpu().numpy().view(np.uint16)
    sin, cos = oracle.rope_tables(128, 128)
    st, ct = torch.from_numpy(sin).to(DEV), torch.from_numpy(cos).to(DEV)
    offs = torch.tensor([0, 11], dtype=torch.int, device=DEV)
    for tag, neox in (("neox", True), ("gptj", False)):
        x = d[f"rope_{tag}_x"].clone()
        ref.rope_(x, st, ct, 17, 8, 128, offs, neox)
        out[f"rope_{tag}_y"] = x.cpu().numpy().view(np.uint16)
    k, v = d["kv_k"], d["kv_v"]
    kq = torch.zeros((2, 9, 8, 64), dtype=torch.uint8, device=DEV)
    ks = torch.zeros((2, 9, 8, 4), dtype=torch.half, device=DEV)
    vq, vs = torch.zeros_like(kq), torch.zeros_like(ks)
    ref.fp16_to_q_kv(k, kq, ks, v, vq, vs, 2, 2, 6, 0, none_tensor, none_tensor, 4)
    ko, vo = torch.zeros_like(k), torch.zeros_like(v)
    ref.q_to_fp16_kv(kq, ko, ks, vq, vo, vs, 2, 2, 6, 0, none_tensor, none_tensor, 4)
    for key, t in (("kq", kq), ("ks", ks), ("vq", vq), ("vs", vs), ("ko", ko), ("vo", vo)):
        out[f"kv_{key}"] = t.cpu().numpy().view(np.uint8)
    os.makedirs(outdir, exist_ok=True)
    np.savez_compressed(os.path.join(outdir, "reference_parity.npz"), **out)
    print("golden parity", len(out), "arrays")
    return 0


def ext_calls(outdir):
    """Every ext_c.<name>(...) call in the reference's hot-path Python files for a Llama-family quantized model."""
    src = os.path.join(REF_ROOT, "exllamav2")
    files = ("linear.py", "cache.py", "rmsnorm.py")
    if not os.path.isdir(src):
        print(f"{src} not found (set EXL2_REFERENCE_ROOT)")
        return 1
    used = set()
    for f in files:
        with open(os.path.join(src, f)) as fh:
            used |= set(re.findall(r"ext_c\.([a-z0-9_]+)\(", fh.read()))
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, "reference_ext_calls.json"), "w") as fh:
        json.dump({"files": [f"exllamav2/{f}" for f in files], "names": sorted(used)}, fh, indent=1)
        fh.write("\n")
    print("ext_c calls", sorted(used))
    return 0


if __name__ == "__main__":
    if sys.argv[1:2] == ["--parity"]:
        sys.exit(parity(sys.argv[2] if len(sys.argv) > 2 else GOLD))
    if sys.argv[1:2] == ["--ext-calls"]:
        sys.exit(ext_calls(sys.argv[2] if len(sys.argv) > 2 else GOLD))
    sys.exit(main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "gpurun_out", "golden")))
