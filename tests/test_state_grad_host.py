"""CPU-only: argument checks of wkv6_train_backward_state_grad, the training backward that takes a gradient for the
final WKV state.  Every bad gT is rejected before anything is launched (no GPU here)."""
import pytest

B, T, C, H = 2, 130, 128, 2
FAKE = 1 << 20                      # a 16-byte aligned fake device address for every other pointer


def _call(lib, gT, gT_f32, C_=C):
    ptrs = [FAKE] * 6               # r, k, v, w, u, s0
    grads = [FAKE] * 8              # gy, gr, gk, gv, gw, gu, gu_total, gs
    return lib.wkv6_train_backward_state_grad(B, T, C_, H, *ptrs, 1, *grads, gT, gT_f32, None, FAKE, 1 << 30, None)


@pytest.mark.parametrize("gT, gT_f32, message", [
    (None, 0, b"gT is NULL"),
    (FAKE + 2, 0, b"gT is not 16-byte aligned"),
    (FAKE + 8, 1, b"gT is not 16-byte aligned"),
    (FAKE, 2, b"gT_f32 = 2"),
    (FAKE, -1, b"gT_f32 = -1"),
])
def test_bad_final_state_gradient_is_rejected_before_any_launch(gT, gT_f32, message):
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    before = lib.wkv6b200_launch_count()
    assert _call(lib, gT, gT_f32) == -1
    assert message in lib.wkv6b200_last_error()
    assert lib.wkv6b200_launch_count() == before


def test_shape_is_checked_first():
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    assert _call(lib, None, 0, C_=100) == -1
    assert b"C == H*64" in lib.wkv6b200_last_error()

