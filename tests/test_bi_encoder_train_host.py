"""CPU-only: argument checks of the two backward entries of bidirectional encoder training,
groupnorm_gate_pair_backward_bf16 and stack_reversed_backward_bf16.  Every misaligned vector argument is rejected,
by name, before any launch; so are C != H*64 and D % 8 != 0."""
import pytest
import torch

pytestmark = pytest.mark.skipif(torch.cuda.is_available(),
                                reason="a library without the check would launch its kernels on the fake addresses")

_ENTRIES = {
    "groupnorm_gate_pair_backward_bf16": (
        ["B", "T", "C", "H", "eps", "gate_act", "y", "y_rev", "rev_idx", "g", "ln_w", "ln_b", "gout", "gy", "gy_rev", "gg",
         "gln_w", "gln_b", "ws", "ws_bytes", "stream"],
        ["y", "y_rev", "g", "ln_w", "ln_b", "gout", "gy", "gy_rev", "gg"]),
    "stack_reversed_backward_bf16": (["B", "T", "D", "gxx", "rev_idx", "gx", "stream"], ["gxx", "gx"]),
}
_SHAPE = {"B": 2, "T": 8, "C": 128, "D": 64, "H": 2, "eps": 1e-5, "gate_act": 1, "ws_bytes": 1 << 30}


def _args(entry, bad=None, **over):
    names = _ENTRIES[entry][0]
    fake = {n: 0x7f0000000000 + 0x100000 * i for i, n in enumerate(names)}
    vals = []
    for n in names:
        if n in over:
            vals.append(over[n])
        elif n in _SHAPE:
            vals.append(_SHAPE[n])
        elif n == "stream":
            vals.append(None)
        else:
            vals.append(fake[n] + (2 if n == bad else 0))
    return vals


@pytest.mark.parametrize("entry", sorted(_ENTRIES))
def test_misaligned_pointers_are_rejected_before_any_launch(entry):
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    names, checked = _ENTRIES[entry]
    assert len(names) == len(_lib.SIGNATURES[entry][1])
    for bad in checked:
        rc = getattr(lib, entry)(*_args(entry, bad))
        msg = lib.wkv6b200_last_error().decode()
        assert rc == -1, (entry, bad, rc, msg)
        assert msg == f"{entry}: {bad} is not 16-byte aligned", (entry, bad, msg)


def test_bad_shapes_are_rejected():
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    e = "groupnorm_gate_pair_backward_bf16"
    assert getattr(lib, e)(*_args(e, C=100)) == -1
    assert b"C == H*64" in lib.wkv6b200_last_error()
    assert getattr(lib, e)(*_args(e, C=128, H=1)) == -1
    assert b"C == H*64" in lib.wkv6b200_last_error()
    assert getattr(lib, e)(*_args(e, ws_bytes=8)) == -1
    assert b"workspace too small" in lib.wkv6b200_last_error()
    assert getattr(lib, e)(*_args(e, gln_b=None)) == -1                 # one affine gradient without the other
    assert b"null pointer" in lib.wkv6b200_last_error()
    e = "stack_reversed_backward_bf16"
    for D in (12, 0, -8):
        assert getattr(lib, e)(*_args(e, D=D)) == -1
        assert b"D % 8 == 0" in lib.wkv6b200_last_error()


def test_empty_problems_are_a_no_op():
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    e = "groupnorm_gate_pair_backward_bf16"
    assert getattr(lib, e)(*_args(e, B=0)) == 0
    assert getattr(lib, e)(*_args(e, T=0, y=None)) == 0
    e = "stack_reversed_backward_bf16"
    assert getattr(lib, e)(*_args(e, B=0, gxx=None)) == 0
