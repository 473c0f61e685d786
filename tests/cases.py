"""Shared seeded test cases (used by the CPU golden tests, the GPU parity tests and oracle/gen_golden.py)."""
import numpy as np

import synth

# name -> kwargs of synth.make_exl2 (small enough that the numpy oracle finishes in milliseconds)
EXL2_CASES = {
    "b4_g128":        dict(K=256, N=128, bits=(4,), bits_prop=(1.0,), group_size=128, seed=11),
    "b4_g32_noperm":  dict(K=128, N=64, bits=(4,), bits_prop=(1.0,), group_size=32, seed=12, perm=False),
    "b54_g64":        dict(K=512, N=128, bits=(5, 4), bits_prop=(0.1, 0.9), group_size=64, seed=13),
    "b43_g128":       dict(K=512, N=192, bits=(4, 3), bits_prop=(0.1, 0.9), group_size=128, seed=14),
    "b32_g64":        dict(K=512, N=64, bits=(3, 2), bits_prop=(0.05, 0.95), group_size=64, seed=15),
    "b865_mixed":     dict(K=512, N=128, bits=(8, 6, 5), bits_prop=(0.05, 0.1, 0.85), group_size=(32, 128, 128), seed=16),
    "b632_mixed":     dict(K=512, N=64, bits=(6, 3, 2), bits_prop=(0.05, 0.2, 0.75), group_size=(32, 64, 64), seed=17),
    "b6_g128_bias":   dict(K=256, N=128, bits=(6,), bits_prop=(1.0,), group_size=128, seed=18, bias=True),
    "b8_g32":         dict(K=128, N=64, bits=(8,), bits_prop=(1.0,), group_size=32, seed=19),
    "b2_g32":         dict(K=128, N=64, bits=(2,), bits_prop=(1.0,), group_size=32, seed=20),
    "b4_n96_ragged":  dict(K=160, N=96, bits=(4,), bits_prop=(1.0,), group_size=64, seed=21),    # N % 64 = 32, last group 32 rows
    "b84_g32_128":    dict(K=384, N=64, bits=(8, 4), bits_prop=(0.05, 0.95), group_size=(32, 128), seed=22),
}

GPTQ_CASES = {
    "gptq_g128":      dict(K=256, N=128, group_size=128, seed=31, act_order=False),
    "gptq_g128_act":  dict(K=512, N=128, group_size=128, seed=32, act_order=True),
    "gptq_g64_act_b": dict(K=256, N=192, group_size=64, seed=33, act_order=True, bias=True),
    "gptq_g32":       dict(K=128, N=72, group_size=32, seed=34, act_order=False),                # N % 64 = 8
}

M_VALUES = (1, 2, 5, 8, 9, 19)


def make_case(name):
    if name in EXL2_CASES:
        return synth.make_exl2(**EXL2_CASES[name])
    return synth.make_gptq(**GPTQ_CASES[name])


def case_shape(name):
    c = EXL2_CASES.get(name) or GPTQ_CASES[name]
    return c["K"], c["N"]


def activations(name, M, seed=0):
    K, _ = case_shape(name)
    rng = np.random.default_rng(1000 + seed + 7 * M + sum(map(ord, name)))
    return rng.normal(0, 1, size=(M, K)).astype(np.float16)


def u16(x):
    return np.ascontiguousarray(x).view(np.uint16)


# cases compared with the reference extension's outputs stored in golden/reference_parity.npz (oracle/gen_golden.py)
REF_GEMM_M = (1, 4, 8, 19)


def ref_cases():
    """The linear cases the reference's kernels support (N a multiple of 32)."""
    return [n for n in list(EXL2_CASES) + list(GPTQ_CASES) if case_shape(n)[1] % 32 == 0]


def ref_ops_inputs():
    """Seeded inputs of the rms_norm / rope / Q4-kv comparison with the reference, in their draw order."""
    rng = np.random.default_rng(123)
    d = {"norm_x": rng.normal(0, 1.5, size=(5, 4096)).astype(np.float16),
         "norm_w": (1 + 0.1 * rng.normal(size=(4096,))).astype(np.float16)}
    for tag in ("neox", "gptj"):
        d[f"rope_{tag}_x"] = rng.normal(0, 1, size=(2, 6, 8 * 128)).astype(np.float16)
    d["kv_k"] = rng.normal(0, 1, size=(2, 9, 8, 128)).astype(np.float16)
    d["kv_v"] = rng.normal(0, 3, size=(2, 9, 8, 128)).astype(np.float16)
    return d


def gptq_4096_row(act_order):
    """BASELINE config 1: a GPTQ 4096 x 4096 g128 matrix and one activation row."""
    w = synth.make_gptq(4096, 4096, 128, seed=0, act_order=act_order)
    a = np.random.default_rng(0).normal(0, 1, size=(1, 4096)).astype(np.float16)
    return w, a
