"""CPU-only: the C-ABI library builds, loads, and exports exactly what include/wkv6_b200.h declares.
No compute calls (no GPU here)."""
import os
import re
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "wkv6_b200.h")).read()
    return set(re.findall(r"WKV6_API\s+[\w \*]+?\b(\w+)\s*\(", src))


def test_header_and_library_agree():
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    declared = _declared()
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    out = subprocess.check_output(["nm", "-D", "--defined-only", _lib.LIB_PATH], text=True)
    exported = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert declared <= exported, declared - exported
    # ... and nothing else: no test kernels, no profiling hooks in the product library
    assert exported <= declared, exported - declared
    assert lib.wkv6b200_abi_version() == 4


def test_argument_validation_without_gpu():
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    # C != H*64 is rejected before anything touches the device
    rc = lib.wkv6_forward(1, 4, 100, 2, None, None, None, None, None, None, None)
    assert rc == -1 and b"C == H*64" in lib.wkv6b200_last_error()
    rc = lib.wkv6_forward(1, 4, 128, 2, None, None, None, None, None, None, None)
    assert rc == -1 and b"null pointer" in lib.wkv6b200_last_error()
    # empty problems are a successful no-op (reference: grid of 0 blocks)
    assert lib.wkv6_forward(0, 4, 128, 2, None, None, None, None, None, None, None) == 0
    assert lib.wkv6_backward_workspace_bytes(2, 8, 128, 2) >= 2 * 8 * 128 * 4


def test_cpu_tensors_fail_loudly():
    import rwkv_lm_ext_b200 as M
    x = torch.zeros(1, 2, 64, dtype=torch.bfloat16)
    u = torch.zeros(1, 64, dtype=torch.bfloat16)
    with pytest.raises(M.Wkv6B200Error):
        M.RUN_CUDA_RWKV6(1, 2, 64, 1, x, x, x, x, u)
    with pytest.raises(AssertionError):          # reference-style dtype assert (src/model.py:195)
        M.RUN_CUDA_RWKV6(1, 2, 64, 1, x.float(), x, x, x, u)


# The memory-bound entries and the arguments they read or write with 16-byte vector accesses (include/wkv6_b200.h).
# Shapes are valid; every pointer argument is a fake, 16-byte aligned device address unless it is the one under test.
_ALIGNED_ENTRIES = {
    "gather_rows_bf16": (["B", "T", "D", "x", "pos", "out", "stream"], ["x", "out"]),
    "pooling_bf16": (["kind", "variant", "B", "T", "D", "x", "actual_len", "out_f32", "stream"], ["x"]),
    "gather_tokens_bf16": (["B", "T", "D", "x", "rev_idx", "out", "stream"], ["x", "out"]),
    "stack_reversed_bf16": (["B", "T", "D", "x", "rev_idx", "out", "stream"], ["x", "out"]),
    "tmix_ddlerp_mix_bf16": (["B", "T", "C", "x", "shift_state", "maa", "m", "out", "stream"],
                             ["x", "shift_state", "maa", "m", "out"]),
    "tmix_ddlerp_lora_bf16": (["B", "T", "C", "R", "x", "shift_state", "maa", "h", "w2", "out", "stream"],
                              ["x", "shift_state", "maa", "h", "w2", "out"]),
    "tmix_shift_lerp_bf16": (["B", "T", "C", "x", "shift_state", "maa_x", "out", "stream"], ["x", "shift_state", "maa_x", "out"]),
    "groupnorm_gate_bf16": (["BT", "C", "H", "eps", "gate_act", "y", "g", "ln_w", "ln_b", "out", "stream"],
                            ["y", "g", "ln_w", "ln_b", "out"]),
    "groupnorm_gate_pair_bf16": (["B", "T", "C", "H", "eps", "gate_act", "y", "y_rev", "rev_idx", "g", "ln_w", "ln_b", "out", "stream"],
                                 ["y", "y_rev", "g", "ln_w", "ln_b", "out"]),
    "tmix_ddlerp_mix_backward_bf16": (["B", "T", "C", "x", "shift_state", "maa", "m", "gxw", "gxk", "gxv", "gxr", "gxg", "gx", "gm",
                                       "gmaa", "gshift", "ws", "ws_bytes", "stream"],
                                      ["x", "shift_state", "maa", "m", "gxw", "gxk", "gxv", "gxr", "gxg", "gx", "gm", "gshift"]),
    "tmix_shift_lerp_backward_bf16": (["B", "T", "C", "x", "shift_state", "maa_x", "gout", "gx", "gmaa_x", "gshift", "ws", "ws_bytes",
                                       "stream"], ["x", "shift_state", "maa_x", "gout", "gx", "gshift"]),
    "groupnorm_gate_backward_bf16": (["BT", "C", "H", "eps", "gate_act", "y", "g", "ln_w", "ln_b", "gout", "gy", "gg", "gln_w", "gln_b",
                                      "ws", "ws_bytes", "stream"], ["y", "g", "ln_w", "ln_b", "gout", "gy", "gg"]),
    "pooling_backward_bf16": (["kind", "variant", "B", "T", "D", "actual_len", "gout_f32", "gx", "stream"], ["gout_f32", "gx"]),
    "scatter_rows_bf16": (["B", "T", "D", "gout", "pos", "gx", "stream"], ["gout", "gx"]),
    "scatter_tokens_bf16": (["B", "T", "D", "gout", "rev_idx", "gx", "stream"], ["gout", "gx"]),
    "cmix_shift_lerp2_bf16": (["B", "T", "C", "x", "shift_state", "maa_kr", "out", "stream"], ["x", "shift_state", "maa_kr", "out"]),
    "cmix_shift_lerp2_backward_bf16": (["B", "T", "C", "x", "shift_state", "maa_kr", "gxk", "gxr", "gx", "gmaa_kr", "gshift", "ws",
                                        "ws_bytes", "stream"], ["x", "shift_state", "gxk", "gxr", "gx", "gshift"]),
    "relu_sq_bf16": (["n", "x", "y", "stream"], ["x", "y"]),
    "relu_sq_backward_bf16": (["n", "x", "gy", "gx", "stream"], ["x", "gy", "gx"]),
    "sigmoid_mul_bf16": (["n", "r", "kv", "out", "stream"], ["r", "kv", "out"]),
    "sigmoid_mul_backward_bf16": (["n", "r", "kv", "gout", "gr", "gkv", "stream"], ["r", "kv", "gout", "gr", "gkv"]),
}
_SHAPE_ARGS = {"B": 2, "T": 8, "C": 64, "D": 64, "H": 1, "R": 32, "BT": 16, "n": 1024, "kind": 0, "variant": 0, "gate_act": 0,
               "eps": 1e-5, "ws_bytes": 1 << 30}


@pytest.mark.skipif(torch.cuda.is_available(),
                    reason="a library without the check would launch its kernels on the fake addresses")
@pytest.mark.parametrize("entry", sorted(_ALIGNED_ENTRIES))
def test_misaligned_pointers_are_rejected_before_any_launch(entry):
    """A contiguous view at an element offset (x[1:]) is 2 bytes off a 16-byte boundary; the 16-byte vector accesses of
    the memory-bound kernels would fault on it.  Every such argument is rejected with WKV6_EINVAL, naming it."""
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    names, checked = _ALIGNED_ENTRIES[entry]
    assert len(names) == len(_lib.SIGNATURES[entry][1])
    fake = {name: 0x7f0000000000 + 0x100000 * i for i, name in enumerate(names) if name not in _SHAPE_ARGS}
    fake["stream"] = None
    for bad in checked:
        args = [_SHAPE_ARGS[n] if n in _SHAPE_ARGS else (fake[n] + 2 if n == bad else fake[n]) for n in names]
        rc = getattr(lib, entry)(*args)
        msg = lib.wkv6b200_last_error().decode()
        assert rc == -1, (entry, bad, rc, msg)
        assert msg == f"{entry}: {bad} is not 16-byte aligned", (entry, bad, msg)


@pytest.mark.skipif(torch.cuda.is_available(),
                    reason="a library without the check would launch its kernels on the fake addresses")
def test_ddlerp_backward_rejects_more_than_int_max_m_rows():
    """The five m planes are read through one tensor map of 5*B rows, an int dimension: B > INT_MAX / 5 is rejected
    before anything is launched, whatever the workspace."""
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    names = _ALIGNED_ENTRIES["tmix_ddlerp_mix_backward_bf16"][0]
    fake = {name: 0x7f0000000000 + 0x100000 * i for i, name in enumerate(names)}
    shape = {"B": (2**31 - 1) // 5 + 1, "T": 1, "C": 8, "ws_bytes": 1 << 62, "stream": None}
    rc = lib.tmix_ddlerp_mix_backward_bf16(*[shape[n] if n in shape else fake[n] for n in names])
    assert rc == -1 and lib.wkv6b200_last_error().decode() == "tmix_ddlerp_mix_backward_bf16: need 5*B <= INT_MAX"


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "rwkv_lm_ext_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in txt.replace("oracle/", "").lower() or f == "_lib.py", f
