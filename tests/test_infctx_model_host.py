"""CPU-only: argument checks of the chunked infctx driver (infctx.infctx_train_step / infctx_forward) and of
wkv6_train_backward_state_grad_ex, the training backward that writes dL/dS_0 in fp32.  Every bad argument is
rejected before anything reaches a device (no GPU here)."""
import pytest
import torch

B, T, C, H = 2, 130, 128, 2
FAKE = 1 << 20                      # a 16-byte aligned fake device address for every other pointer


def _model(layers=2):
    from rwkv_lm_ext_b200 import sft
    return sft.RwkvSft(layers=layers, D=C, H=H, ffn=2 * C, vocab=64, train_type="full")


def _ids(b=B, t=T):
    return torch.zeros(b, t, dtype=torch.long)


@pytest.mark.parametrize("chunk_ctx", [0, -4, 2.5, None])
def test_bad_chunk_ctx(chunk_ctx):
    from rwkv_lm_ext_b200.infctx import infctx_train_step
    with pytest.raises(ValueError, match="chunk_ctx"):
        infctx_train_step(_model(), _ids(), _ids(), chunk_ctx)


@pytest.mark.parametrize("idx_shape, tgt_shape", [((B, T), (B, T - 1)), ((B, T), (B + 1, T)), ((T,), (T,))])
def test_idx_and_targets_must_agree(idx_shape, tgt_shape):
    from rwkv_lm_ext_b200.infctx import infctx_train_step
    idx, tgt = torch.zeros(idx_shape, dtype=torch.long), torch.zeros(tgt_shape, dtype=torch.long)
    with pytest.raises(ValueError, match="idx and targets"):
        infctx_train_step(_model(), idx, tgt, 64)


@pytest.mark.parametrize("layers, b, c, h, what", [
    (3, B, C, H, "wkv_states"),         # one layer too many
    (1, B, C, H, "wkv_states"),         # one too few
    (2, B + 1, C, H, "wkv_states"),     # batch
    (2, B, C, H, None),                 # shift states of the wrong width (built below)
])
def test_states_must_fit_the_model(layers, b, c, h, what):
    from rwkv_lm_ext_b200.infctx import BlockStateList, infctx_forward, infctx_train_step
    st = BlockStateList.create(layers, b, c, h, "cpu", torch.bfloat16, wkv_dtype=torch.float32)
    if what is None:
        st = BlockStateList(torch.zeros(layers, 2, b, c + 64, dtype=torch.bfloat16), st.wkv_states)
    with pytest.raises(ValueError, match=what or "shift_states"):
        infctx_train_step(_model(), _ids(), _ids(), 64, states=st)
    with pytest.raises(ValueError, match=what or "shift_states"):
        infctx_forward(_model(), _ids(), st)


def test_states_must_be_a_block_state_list():
    from rwkv_lm_ext_b200.infctx import infctx_train_step
    with pytest.raises(TypeError, match="BlockStateList"):
        infctx_train_step(_model(), _ids(), _ids(), 64, states=(torch.zeros(1), torch.zeros(1)))


def _call_ex(lib, gT, gT_f32, gs, gs_f32, C_=C):
    ptrs = [FAKE] * 6               # r, k, v, w, u, s0
    grads = [FAKE] * 7              # gy, gr, gk, gv, gw, gu, gu_total
    return lib.wkv6_train_backward_state_grad_ex(B, T, C_, H, *ptrs, 1, *grads, gT, gT_f32, gs, gs_f32, None, FAKE,
                                                 1 << 30, None)


@pytest.mark.parametrize("gT, gT_f32, gs, gs_f32, message", [
    (FAKE, 0, FAKE, 2, b"gs_f32 = 2"),
    (FAKE, 0, FAKE, -1, b"gs_f32 = -1"),
    (None, 0, None, 1, b"gs is NULL"),
    (FAKE, 1, None, 0, b"gs is NULL"),
    (FAKE, 0, FAKE + 4, 1, b"gs is not 16-byte aligned"),
    (None, 0, FAKE + 2, 0, b"gs is not 16-byte aligned"),
    (FAKE + 8, 1, FAKE, 1, b"gT is not 16-byte aligned"),
    (FAKE, 2, FAKE, 1, b"gT_f32 = 2"),
])
def test_bad_state_gradient_arguments_are_rejected_before_any_launch(gT, gT_f32, gs, gs_f32, message):
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    before = lib.wkv6b200_launch_count()
    assert _call_ex(lib, gT, gT_f32, gs, gs_f32) == -1
    assert message in lib.wkv6b200_last_error()
    assert lib.wkv6b200_launch_count() == before


def test_shape_is_checked_first():
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    assert _call_ex(lib, None, 0, None, 2, C_=100) == -1
    assert b"C == H*64" in lib.wkv6b200_last_error()
