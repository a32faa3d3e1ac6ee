"""The RWKV-6 channel-mix layer on fused elementwise kernels (SURVEY.md section 8(f) rank 2).

`cmix_x060_forward(layer, x[, last_state])` computes `RWKV_CMix_x060.forward` (src/model.py:635-644; the
infctx flavour :804-812 when a `ChannelMixState` / shift tensor is given) on any module with the
reference's parameter names `time_maa_k`, `time_maa_r`, `key`, `receptance`, `value`:

    xk, xr = x + (shift(x) - x) * time_maa_{k,r}       one kernel, x read once
    k      = relu(key(xk)) ** 2                         one kernel
    out    = sigmoid(receptance(xr)) * value(k)         one kernel

The forwards are bit-identical to the eager bf16 chain (packed bf16 arithmetic, non-contracting); every
piece is a `torch.autograd.Function`.
"""
import torch

from . import _lib
from ._lib import check, ptr, stream_of
from .heads import _bf16_param, _cuda, _dense, _needs_grad, _ws


class _ShiftLerp2(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, shift_state, maa_kr):
        ctx.save_for_backward(x, shift_state, maa_kr)
        return tuple(_shift_lerp2_fwd(x, shift_state, maa_kr).unbind(0))

    @staticmethod
    def backward(ctx, gxk, gxr):
        x, shift_state, maa_kr = ctx.saved_tensors
        lib = _lib.load()
        B, T, C = x.shape
        gxk = torch.zeros_like(x) if gxk is None else _dense(gxk)
        gxr = torch.zeros_like(x) if gxr is None else _dense(gxr)
        gx = torch.empty_like(x)
        gmaa = torch.empty(2, C, dtype=torch.float32, device=x.device) if ctx.needs_input_grad[2] else None
        gshift = torch.empty_like(shift_state) if shift_state is not None else None
        ws = _ws(lib, B, T, C, 3, x.device)
        check(lib.cmix_shift_lerp2_backward_bf16(B, T, C, ptr(x), ptr(shift_state), ptr(maa_kr), ptr(gxk), ptr(gxr), ptr(gx),
                                                 ptr(gmaa), ptr(gshift), ptr(ws), ws.numel(), stream_of(x)),
              "cmix_shift_lerp2_backward_bf16")
        return gx, gshift, (gmaa.to(maa_kr.dtype) if gmaa is not None else None)


def _shift_lerp2_fwd(x, shift_state, maa_kr):
    B, T, C = x.shape
    out = torch.empty(2, B, T, C, dtype=torch.bfloat16, device=x.device)
    check(_lib.load().cmix_shift_lerp2_bf16(B, T, C, ptr(x), ptr(shift_state), ptr(maa_kr), ptr(out), stream_of(x)),
          "cmix_shift_lerp2_bf16")
    return out


def cmix_shift_lerp2(x, maa_k, maa_r, shift_state=None):
    """(xk, xr) of src/model.py:637-639."""
    _cuda(x)
    assert x.dtype == torch.bfloat16
    x = _dense(x)
    C = x.shape[-1]
    maa_kr = _bf16_param(torch.cat([maa_k.reshape(1, C), maa_r.reshape(1, C)], 0))      # (two [C] rows: a 3 us launch)
    shift_state = _bf16_param(shift_state)
    if _needs_grad(x, maa_kr, shift_state):
        return _ShiftLerp2.apply(x, shift_state, maa_kr)
    return tuple(_shift_lerp2_fwd(x, shift_state, maa_kr).unbind(0))


class _ReluSq(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        y = torch.empty_like(x)
        check(_lib.load().relu_sq_bf16(x.numel(), ptr(x), ptr(y), stream_of(x)), "relu_sq_bf16")
        return y

    @staticmethod
    def backward(ctx, gy):
        (x,) = ctx.saved_tensors
        gy = _dense(gy)
        gx = torch.empty_like(x)
        check(_lib.load().relu_sq_backward_bf16(x.numel(), ptr(x), ptr(gy), ptr(gx), stream_of(x)), "relu_sq_backward_bf16")
        return gx


def relu_sq(x):
    """torch.relu(x) ** 2  (src/model.py:642)."""
    _cuda(x)
    assert x.dtype == torch.bfloat16
    x = _dense(x)
    if x.numel() % 8:
        return torch.relu(x) ** 2
    return _ReluSq.apply(x)


class _SigmoidMul(torch.autograd.Function):
    @staticmethod
    def forward(ctx, r, kv):
        ctx.save_for_backward(r, kv)
        out = torch.empty_like(r)
        check(_lib.load().sigmoid_mul_bf16(r.numel(), ptr(r), ptr(kv), ptr(out), stream_of(r)), "sigmoid_mul_bf16")
        return out

    @staticmethod
    def backward(ctx, gout):
        r, kv = ctx.saved_tensors
        gout = _dense(gout)
        gr, gkv = torch.empty_like(r), torch.empty_like(kv)
        check(_lib.load().sigmoid_mul_backward_bf16(r.numel(), ptr(r), ptr(kv), ptr(gout), ptr(gr), ptr(gkv), stream_of(r)),
              "sigmoid_mul_backward_bf16")
        return gr, gkv


def sigmoid_mul(r, kv):
    """torch.sigmoid(r) * kv  (src/model.py:644)."""
    _cuda(r)
    assert r.dtype == torch.bfloat16 and kv.dtype == torch.bfloat16 and r.shape == kv.shape
    r, kv = _dense(r), _dense(kv)
    if r.numel() % 8:
        return torch.sigmoid(r) * kv
    return _SigmoidMul.apply(r, kv)


def cmix_x060_forward(layer, x, last_state=None):
    """Drop-in for RWKV_CMix_x060.forward; with `last_state` (a ChannelMixState or the [B,C] shift tensor)
    the infctx flavour, returning (out, new_state)."""
    shift = None
    if last_state is not None:
        shift = last_state.shift_state if hasattr(last_state, "shift_state") else last_state
    xk, xr = cmix_shift_lerp2(x, layer.time_maa_k, layer.time_maa_r, shift)
    out = sigmoid_mul(layer.receptance(xr), layer.value(relu_sq(layer.key(xk))))
    if last_state is None:
        return out
    new = x[:, -1]
    return out, (type(last_state)(new) if hasattr(last_state, "shift_state") else new)
