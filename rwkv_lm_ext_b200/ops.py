"""The reference's WKV operator surface, backed by libwkv6_b200.so.

Same names, positional signatures, dtype/contiguity asserts and return conventions as
  * src/model.py:83-235      WKV_6, WKV_6STATE (states / infctx), RUN_CUDA_RWKV6, RUN_CUDA_RWKV6_STATE
  * src/model_run.py:49-76   RWKV_6, RUN_RWKV_6
  * cuda/wkv6_bi.py:13-60    WKV_6_BI, RUN_CUDA_RWKV6(B,T,C,H,mask,...)
so that ``src.model.RUN_CUDA_RWKV6 = rwkv_lm_ext_b200.RUN_CUDA_RWKV6`` (see ``install``) redirects every
Tmix layer of the unmodified reference models.  Host code is PyTorch (allocation, autograd
plumbing, streams); all arithmetic happens in the C-ABI library.  No CPU fallback.
"""
import ctypes
import os

import torch

from . import _lib
from ._lib import check, ptr, stream_of

HEAD_SIZE = 64  # RWKV_HEAD_SIZE_A, hard-wired like the reference (src/model_run.py:15)


def _assert_bf16_contig(*ts):
    for t in ts:
        assert t.dtype == torch.bfloat16
        assert t.is_contiguous()


def _require_cuda(t):
    _lib.require_current_device(t)


def _workspace(lib, B, T, C, H, device):
    n = lib.wkv6_backward_workspace_bytes(B, T, C, H)
    return torch.empty(max(n, 1), dtype=torch.uint8, device=device), n


def _train_forward(ctx, lib, B, T, C, H, r, k, v, w, u, s0, s0_batched, sT, y):
    """Forward of the training pair (include/wkv6_b200.h): when a gradient will be asked for, the
    kernel also leaves the bf16 chunk-start states in ``ctx.saved_state`` -- kept next to
    save_for_backward's r,k,v,w,u like the reference keeps its inputs (src/model.py:203) -- so that
    backward does not re-run the recurrence."""
    saved = None
    if any(ctx.needs_input_grad):
        saved = torch.empty(lib.wkv6_saved_bytes(B, T, C, H), dtype=torch.uint8, device=r.device)
    valid = ctypes.c_int(0)
    s0_f32 = int(s0 is not None and s0.dtype == torch.float32)
    sT_f32 = int(sT is not None and sT.dtype == torch.float32)
    check(lib.wkv6_train_forward(B, T, C, H, ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(s0), int(s0_batched),
                                 s0_f32, ptr(sT), sT_f32, ptr(y), ptr(saved), ctypes.byref(valid), stream_of(r)),
          "wkv6_train_forward")
    ctx.saved_state = saved if valid.value else None
    if _diag["collect"] and ctx.saved_state is not None:
        _diag["streams"] += B * H


# Diagnostics: how many (b,h) streams of the training forwards left the tensor-core kernels for the exact SIMT route.
# None does: the block references and the decay floor cover every decay (DESIGN.md 4.0), and only an fp32 decay that is
# not a bf16 logit -- never the training pair's raw logits -- is handed to the exact kernels.
_diag = {"collect": False, "streams": 0}


class exact_route_report:
    """with exact_route_report() as rep: ...training forwards...;  rep.streams() -> (flagged, total)"""

    def __enter__(self):
        _diag["collect"], _diag["streams"] = True, 0
        return self

    def __exit__(self, *exc):
        self._streams = _diag["streams"]
        _diag["collect"], _diag["streams"] = False, 0
        return False

    def streams(self):
        return 0, self._streams


def _train_backward(ctx, lib, B, T, C, H, r, k, v, w, u, s0, s0_batched, gy, gr, gk, gv, gw, gu, gs, gT=None):
    """Returns gu summed over the batch rows (src/model.py:232 `torch.sum(gu, 0)`), computed by the library.
    gT: None, or the gradient of the final state (bf16/fp32 [B,H,64,64], contiguous, 16-byte aligned)."""
    saved = ctx.saved_state
    n = lib.wkv6_train_backward_workspace_bytes(B, T, C, H, int(saved is not None))
    ws = torch.empty(max(n, 1), dtype=torch.uint8, device=gy.device)
    gu_total = torch.empty((C,), device=gy.device, dtype=torch.bfloat16)
    head = (B, T, C, H, ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(s0), int(s0_batched),
            ptr(gy), ptr(gr), ptr(gk), ptr(gv), ptr(gw), ptr(gu), ptr(gu_total), ptr(gs))
    tail = (ptr(saved), ptr(ws), n, stream_of(gy))
    if gT is None:
        check(lib.wkv6_train_backward(*head, *tail), "wkv6_train_backward")
    else:
        check(lib.wkv6_train_backward_state_grad(*head, ptr(gT), int(gT.dtype == torch.float32), *tail),
              "wkv6_train_backward_state_grad")
    return gu_total


# --------------------------------------------------------------------------------------------
# WKV_6  (src/model.py:191-235)
# --------------------------------------------------------------------------------------------
class WKV_6(torch.autograd.Function):
    """y = WKV6(r,k,v,w,u), S_0 = 0.  The reference materialises ew = -exp(w.float()) in PyTorch
    (src/model.py:210) and hands it to the kernel; here the kernel reads the raw bf16 logits."""

    @staticmethod
    def forward(ctx, B, T, C, H, r, k, v, w, u):
        with torch.no_grad():
            _assert_bf16_contig(r, k, v, w, u)
            assert HEAD_SIZE == C // H
            _require_cuda(r)
            ctx.B, ctx.T, ctx.C, ctx.H = B, T, C, H
            ctx.save_for_backward(r, k, v, w, u)
            y = torch.empty((B, T, C), device=r.device, dtype=torch.bfloat16, memory_format=torch.contiguous_format)
            lib = _lib.load()
            _train_forward(ctx, lib, B, T, C, H, r, k, v, w, u, None, False, None, y)
            return y

    @staticmethod
    def backward(ctx, gy):
        with torch.no_grad():
            assert gy.dtype == torch.bfloat16
            B, T, C, H = ctx.B, ctx.T, ctx.C, ctx.H
            gy = gy.contiguous()
            r, k, v, w, u = ctx.saved_tensors
            gr, gk, gv, gw = (torch.empty((B, T, C), device=gy.device, dtype=torch.bfloat16) for _ in range(4))
            gu = torch.empty((B, C), device=gy.device, dtype=torch.bfloat16)
            lib = _lib.load()
            gu = _train_backward(ctx, lib, B, T, C, H, r, k, v, w, u, None, False, gy, gr, gk, gv, gw, gu, None)
            gu = gu.view(H, C // H)                        # src/model.py:232 (the sum over B happens in the library)
            return (None, None, None, None, gr, gk, gv, gw, gu)


def RUN_CUDA_RWKV6(B, T, C, H, r, k, v, w, u):
    """src/model.py:235 (also imported late by src/model_ext.py:353,432 and src/model_encoder_run.py:88)."""
    return WKV_6.apply(B, T, C, H, r, k, v, w, u)


# --------------------------------------------------------------------------------------------
# WKV_6STATE, "states" flavour (src/model.py:137-185): s = time_state [H,64,64], shared, trainable
# --------------------------------------------------------------------------------------------
class WKV_6STATE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, B, T, C, H, r, k, v, w, u, s):
        with torch.no_grad():
            _assert_bf16_contig(r, k, v, w, u, s)
            assert HEAD_SIZE == C // H
            _require_cuda(r)
            assert tuple(s.shape) == (H, HEAD_SIZE, HEAD_SIZE)
            ctx.B, ctx.T, ctx.C, ctx.H = B, T, C, H
            ctx.save_for_backward(r, k, v, w, u, s)
            y = torch.empty((B, T, C), device=r.device, dtype=torch.bfloat16, memory_format=torch.contiguous_format)
            lib = _lib.load()
            _train_forward(ctx, lib, B, T, C, H, r, k, v, w, u, s, False, None, y)
            return y

    @staticmethod
    def backward(ctx, gy):
        with torch.no_grad():
            assert gy.dtype == torch.bfloat16
            B, T, C, H = ctx.B, ctx.T, ctx.C, ctx.H
            gy = gy.contiguous()
            r, k, v, w, u, s = ctx.saved_tensors
            gr, gk, gv, gw = (torch.empty((B, T, C), device=gy.device, dtype=torch.bfloat16) for _ in range(4))
            gu = torch.empty((B, C), device=gy.device, dtype=torch.bfloat16)
            gs = torch.empty((B, H, C // H, C // H), device=gy.device, dtype=torch.bfloat16)
            lib = _lib.load()
            gu = _train_backward(ctx, lib, B, T, C, H, r, k, v, w, u, s, False, gy, gr, gk, gv, gw, gu, gs)
            gu = gu.view(H, C // H)                                # src/model.py:181 (summed over B in the library)
            gs = torch.sum(gs, 0).view(H, C // H, C // H)          # src/model.py:182
            return (None, None, None, None, gr, gk, gv, gw, gu, gs)


# --------------------------------------------------------------------------------------------
# WKV_6STATE, "infctx" flavour (src/model.py:83-132): s [B,H,64,64], final state written in place
# --------------------------------------------------------------------------------------------
class WKV_6STATE_INFCTX(torch.autograd.Function):
    @staticmethod
    def forward(ctx, B, T, C, H, r, k, v, w, u, s):
        with torch.no_grad():
            _assert_bf16_contig(r, k, v, w, u)
            assert s.dtype in (torch.bfloat16, torch.float32)      # fp32 carry is an extension
            assert s.is_contiguous()
            assert HEAD_SIZE == C // H
            _require_cuda(r)
            assert tuple(s.shape) == (B, H, HEAD_SIZE, HEAD_SIZE)
            ctx.B, ctx.T, ctx.C, ctx.H = B, T, C, H
            # the reference saves `s` and then overwrites it (src/model.py:104-106), so its backward
            # sees the FINAL state; keep the initial one instead (SURVEY.md 2.3)
            s_init = s.to(torch.bfloat16, copy=True)
            ctx.save_for_backward(r, k, v, w, u, s_init)
            y = torch.empty((B, T, C), device=r.device, dtype=torch.bfloat16, memory_format=torch.contiguous_format)
            lib = _lib.load()
            _train_forward(ctx, lib, B, T, C, H, r, k, v, w, u, s, True, s, y)
            ctx.mark_dirty(s)
            ctx.s_dtype = s.dtype
            return y, s

    @staticmethod
    def backward(ctx, gy, _gs_final):
        with torch.no_grad():
            assert gy.dtype == torch.bfloat16
            B, T, C, H = ctx.B, ctx.T, ctx.C, ctx.H
            gy = gy.contiguous()
            r, k, v, w, u, s = ctx.saved_tensors
            gr, gk, gv, gw = (torch.empty((B, T, C), device=gy.device, dtype=torch.bfloat16) for _ in range(4))
            gu = torch.empty((B, C), device=gy.device, dtype=torch.bfloat16)
            gs = torch.empty((B, H, C // H, C // H), device=gy.device, dtype=torch.bfloat16)
            lib = _lib.load()
            gu = _train_backward(ctx, lib, B, T, C, H, r, k, v, w, u, s, True, gy, gr, gk, gv, gw, gu, gs)
            gu = gu.view(H, C // H)
            # per-sample state: its gradient is per sample too.  (The reference sums gs over the
            # batch into [H,64,64] even here, src/model.py:128 -- a shape that cannot flow back
            # into a [B,H,64,64] leaf; truncated BPTT: the final state gets no gradient.)
            return (None, None, None, None, gr, gk, gv, gw, gu, gs.to(ctx.s_dtype))


class WKV_6STATE_BPTT(torch.autograd.Function):
    """The infctx operator with gradients through the carried state: out of place (``s`` is read, never written;
    ``s_final`` is a new tensor with the dtype of ``s``, bf16 or the fp32 carry), and the gradient of ``s_final``
    flows back into r, k, v, w, u and ``s``.  Chunked long-context training then computes the gradients of one
    pass over the whole sequence.  A ``s_final`` that feeds nothing (gradient None) runs the backward of
    WKV_6STATE_INFCTX."""

    @staticmethod
    def forward(ctx, B, T, C, H, r, k, v, w, u, s):
        with torch.no_grad():
            _assert_bf16_contig(r, k, v, w, u)
            assert s.dtype in (torch.bfloat16, torch.float32)
            assert s.is_contiguous()
            assert HEAD_SIZE == C // H
            _require_cuda(r)
            assert tuple(s.shape) == (B, H, HEAD_SIZE, HEAD_SIZE)
            ctx.B, ctx.T, ctx.C, ctx.H = B, T, C, H
            ctx.save_for_backward(r, k, v, w, u, s.to(torch.bfloat16))
            y = torch.empty((B, T, C), device=r.device, dtype=torch.bfloat16, memory_format=torch.contiguous_format)
            s_final = torch.empty_like(s, memory_format=torch.contiguous_format)
            lib = _lib.load()
            _train_forward(ctx, lib, B, T, C, H, r, k, v, w, u, s, True, s_final, y)
            ctx.s_dtype = s.dtype
            return y, s_final

    @staticmethod
    def backward(ctx, gy, gs_final):
        with torch.no_grad():
            B, T, C, H = ctx.B, ctx.T, ctx.C, ctx.H
            r, k, v, w, u, s = ctx.saved_tensors
            if gy is None:                                         # only the final state feeds the loss
                gy = torch.zeros((B, T, C), device=r.device, dtype=torch.bfloat16)
            assert gy.dtype == torch.bfloat16
            gy = gy.contiguous()
            gr, gk, gv, gw = (torch.empty((B, T, C), device=gy.device, dtype=torch.bfloat16) for _ in range(4))
            gu = torch.empty((B, C), device=gy.device, dtype=torch.bfloat16)
            gs = torch.empty((B, H, C // H, C // H), device=gy.device, dtype=torch.bfloat16)
            gT = None
            if gs_final is not None:
                gT = gs_final.contiguous()
                assert gT.dtype in (torch.bfloat16, torch.float32) and tuple(gT.shape) == (B, H, HEAD_SIZE, HEAD_SIZE)
                if gT.data_ptr() % 16:                             # the library reads it with 16-byte accesses
                    gT = gT.clone()
            lib = _lib.load()
            gu = _train_backward(ctx, lib, B, T, C, H, r, k, v, w, u, s, True, gy, gr, gk, gv, gw, gu, gs, gT)
            gu = gu.view(H, C // H)
            return (None, None, None, None, gr, gk, gv, gw, gu, gs.to(ctx.s_dtype))


def RUN_CUDA_RWKV6_STATE_BPTT(B, T, C, H, r, k, v, w, u, s):
    """(y, s_final) of the infctx operator, differentiable through s_final (WKV_6STATE_BPTT); ``s`` is not modified."""
    return WKV_6STATE_BPTT.apply(B, T, C, H, r, k, v, w, u, s)


def RUN_CUDA_RWKV6_STATE(B, T, C, H, r, k, v, w, u, s):
    """src/model.py:184 (states: returns y) and src/model.py:130-132 (infctx: returns (y, s)).
    The reference picks one at import time from RWKV_TRAIN_TYPE; here the environment variable is
    honoured when set and otherwise the rank of ``s`` decides ([H,64,64] vs [B,H,64,64])."""
    mode = os.environ.get("RWKV_TRAIN_TYPE", "")
    if mode == "infctx" or (mode != "states" and s.dim() == 4):
        return WKV_6STATE_INFCTX.apply(B, T, C, H, r, k, v, w, u, s)
    return WKV_6STATE.apply(B, T, C, H, r, k, v, w, u, s)


# --------------------------------------------------------------------------------------------
# RWKV_6 inference op (src/model_run.py:49-76)
# --------------------------------------------------------------------------------------------
class RWKV_6(torch.autograd.Function):
    @staticmethod
    def forward(ctx, B, T, C, H, state, r, k, v, w, u):
        with torch.no_grad():
            assert HEAD_SIZE == C // H
            ctx.B, ctx.T, ctx.C, ctx.H = B, T, C, H
            assert state.dtype == torch.float32
            assert state.numel() == B * H * HEAD_SIZE * HEAD_SIZE, "state must be [B,H,64,64] ([H,64,64] when B == 1)"
            assert r.is_contiguous() and k.is_contiguous() and v.is_contiguous()
            assert w.is_contiguous() and u.is_contiguous() and state.is_contiguous()
            _require_cuda(r)
            y = torch.empty((B, T, C), device=w.device, dtype=r.dtype, memory_format=torch.contiguous_format)
            lib = _lib.load()
            if r.dtype == torch.bfloat16 and all(t.dtype == torch.bfloat16 for t in (k, v, w, u)):
                # bf16 models: the kernels read the raw logits themselves -- no exp(-exp(w.float())) passes
                check(lib.rwkv6_forward_raww(B, T, C, H, ptr(state), ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(y),
                                             stream_of(r)), "rwkv6_forward_raww")
            else:
                # the reference computes eew = exp(-exp(w.float())) in PyTorch first (src/model_run.py:64)
                eew = torch.exp(-torch.exp(w.float())).contiguous()
                code = {torch.bfloat16: 0, torch.float16: 1, torch.float32: 2}[r.dtype]
                check(lib.rwkv6_forward(code, B, T, C, H, ptr(state), ptr(r), ptr(k), ptr(v), ptr(eew), ptr(u),
                                        ptr(y), stream_of(r)), "rwkv6_forward")
            ctx.mark_dirty(state)
            return y, state


def RUN_RWKV_6(B, T, C, H, state, r, k, v, w, u):
    """src/model_run.py:75-76: returns (y [B,T,C], state); ``state`` fp32 [(B,)H,64,64] (value,key)
    is updated in place; r,k,v,w,u in the model dtype, w = raw decay logits."""
    return RWKV_6.apply(B, T, C, H, state, r, k, v, w, u)


# --------------------------------------------------------------------------------------------
# WKV_6_BI (cuda/wkv6_bi.py:13-60)
# --------------------------------------------------------------------------------------------
class WKV_6_BI(torch.autograd.Function):
    @staticmethod
    def forward(ctx, B, T, C, H, mask, r, k, v, w, u):
        with torch.no_grad():
            _assert_bf16_contig(r, k, v, w, u)
            assert mask.dtype == torch.int
            assert mask.is_contiguous()
            assert HEAD_SIZE == C // H
            _require_cuda(r)
            ctx.B, ctx.T, ctx.C, ctx.H = B, T, C, H
            ctx.mask = mask
            ctx.save_for_backward(r, k, v, w, u)
            y = torch.empty((B, T, C), device=r.device, dtype=torch.bfloat16, memory_format=torch.contiguous_format)
            lib = _lib.load()
            check(lib.wkv6_bi_forward_raww(B, T, C, H, ptr(mask), ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(y),
                                           stream_of(r)), "wkv6_bi_forward_raww")
            return y

    @staticmethod
    def backward(ctx, gy):
        with torch.no_grad():
            assert gy.dtype == torch.bfloat16
            B, T, C, H = ctx.B, ctx.T, ctx.C, ctx.H
            gy = gy.contiguous()
            r, k, v, w, u = ctx.saved_tensors
            gr, gk, gv, gw = (torch.empty((B, T, C), device=gy.device, dtype=torch.bfloat16) for _ in range(4))
            gu = torch.empty((B, C), device=gy.device, dtype=torch.bfloat16)
            lib = _lib.load()
            ws, n = _workspace(lib, B, T, C, H, gy.device)
            check(lib.wkv6_bi_backward_raww(B, T, C, H, ptr(ctx.mask), ptr(r), ptr(k), ptr(v), ptr(w), ptr(u),
                                            ptr(gy), ptr(gr), ptr(gk), ptr(gv), ptr(gw), ptr(gu), ptr(ws), n,
                                            stream_of(gy)), "wkv6_bi_backward_raww")
            gu = torch.sum(gu, 0).view(H, C // H)
            return (None, None, None, None, None, gr, gk, gv, gw, gu)


def RUN_CUDA_RWKV6_BI(B, T, C, H, mask, r, k, v, w, u):
    """cuda/wkv6_bi.py:59-60 (there it is also called RUN_CUDA_RWKV6, with the extra mask argument)."""
    return WKV_6_BI.apply(B, T, C, H, mask, r, k, v, w, u)


# --------------------------------------------------------------------------------------------
# the reference's NATIVE surface: objects with the pybind signatures of cuda/*_op.cpp, for callers
# (or an unmodified torch.autograd.Function from the reference) that hold pre-allocated outputs
# --------------------------------------------------------------------------------------------
class _NativeWkv6:
    """wkv6_cuda.forward / backward of cuda/wkv6_op.cpp:8-17 (w = fp32 -exp(w))."""

    @staticmethod
    def forward(B, T, C, H, r, k, v, w, u, y):
        check(_lib.load().wkv6_forward(B, T, C, H, ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(y), stream_of(r)),
              "wkv6_forward")

    @staticmethod
    def backward(B, T, C, H, r, k, v, w, u, gy, gr, gk, gv, gw, gu):
        lib = _lib.load()
        ws, n = _workspace(lib, B, T, C, H, r.device)
        check(lib.wkv6_backward(B, T, C, H, ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(gy), ptr(gr), ptr(gk),
                                ptr(gv), ptr(gw), ptr(gu), ptr(ws), n, stream_of(r)), "wkv6_backward")


class _NativeWkv6State:
    """wkv6state_cuda.forward / backward of cuda/wkv6state_op.cpp:8-16 (s [H,64,64])."""

    @staticmethod
    def forward(B, T, C, H, r, k, v, w, u, s, y):
        check(_lib.load().wkv6state_forward(B, T, C, H, ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(s), ptr(y),
                                            stream_of(r)), "wkv6state_forward")

    @staticmethod
    def backward(B, T, C, H, r, k, v, w, u, s, gy, gr, gk, gv, gw, gu, gs):
        lib = _lib.load()
        ws, n = _workspace(lib, B, T, C, H, r.device)
        check(lib.wkv6state_backward(B, T, C, H, ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(s), ptr(gy), ptr(gr),
                                     ptr(gk), ptr(gv), ptr(gw), ptr(gu), ptr(gs), ptr(ws), n, stream_of(r)),
              "wkv6state_backward")


class _NativeWkv6Infctx:
    """wkv6infctx forward / backward of cuda/wkv6infctx_op.cpp:8-16 (s [B,H,64,64], in place)."""

    @staticmethod
    def forward(B, T, C, H, r, k, v, w, u, s, y):
        check(_lib.load().wkv6infctx_forward(B, T, C, H, ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(s), ptr(y),
                                             stream_of(r)), "wkv6infctx_forward")

    @staticmethod
    def backward(B, T, C, H, r, k, v, w, u, s, gy, gr, gk, gv, gw, gu, gs):
        lib = _lib.load()
        ws, n = _workspace(lib, B, T, C, H, r.device)
        check(lib.wkv6infctx_backward(B, T, C, H, ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(s), ptr(gy), ptr(gr),
                                      ptr(gk), ptr(gv), ptr(gw), ptr(gu), ptr(gs), ptr(ws), n, stream_of(r)),
              "wkv6infctx_backward")


class _NativeWkv6Bi:
    """wkv6_bi forward / backward of cuda/wkv6_bi_op.cpp:8-16 (mask int32 [B,T], w = fp32 -exp(w))."""

    @staticmethod
    def forward(B, T, C, H, mask, r, k, v, w, u, y):
        check(_lib.load().wkv6_bi_forward(B, T, C, H, ptr(mask), ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(y),
                                          stream_of(r)), "wkv6_bi_forward")

    @staticmethod
    def backward(B, T, C, H, mask, r, k, v, w, u, gy, gr, gk, gv, gw, gu):
        lib = _lib.load()
        ws, n = _workspace(lib, B, T, C, H, r.device)
        check(lib.wkv6_bi_backward(B, T, C, H, ptr(mask), ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(gy), ptr(gr),
                                   ptr(gk), ptr(gv), ptr(gw), ptr(gu), ptr(ws), n, stream_of(r)), "wkv6_bi_backward")


class _NativeRwkv6:
    """rwkv6.forward_bf16 / _fp16 / _fp32 of cuda/rwkv6_op.cpp:12-34 (w = fp32 decay)."""

    @staticmethod
    def _fwd(code, B, T, C, H, state, r, k, v, w, u, y):
        check(_lib.load().rwkv6_forward(code, B, T, C, H, ptr(state), ptr(r), ptr(k), ptr(v), ptr(w), ptr(u), ptr(y),
                                        stream_of(r)), "rwkv6_forward")

    @staticmethod
    def forward_bf16(B, T, C, H, state, r, k, v, w, u, y):
        _NativeRwkv6._fwd(0, B, T, C, H, state, r, k, v, w, u, y)

    @staticmethod
    def forward_fp16(B, T, C, H, state, r, k, v, w, u, y):
        _NativeRwkv6._fwd(1, B, T, C, H, state, r, k, v, w, u, y)

    @staticmethod
    def forward_fp32(B, T, C, H, state, r, k, v, w, u, y):
        _NativeRwkv6._fwd(2, B, T, C, H, state, r, k, v, w, u, y)


wkv6_cuda = _NativeWkv6
wkv6state_cuda = _NativeWkv6State
wkv6infctx_cuda = _NativeWkv6Infctx
wkv6_bi_cuda = _NativeWkv6Bi
rwkv6 = _NativeRwkv6


def install(module, train_type=None):
    """Point an already-imported reference module (src.model, src.model_bi, src.model_run, ...) at
    these operators: the one-line integration of INTEGRATION.md."""
    if hasattr(module, "RUN_CUDA_RWKV6"):
        module.RUN_CUDA_RWKV6 = RUN_CUDA_RWKV6
    if hasattr(module, "RUN_CUDA_RWKV6_STATE") or train_type in ("states", "infctx"):
        module.RUN_CUDA_RWKV6_STATE = RUN_CUDA_RWKV6_STATE
    if hasattr(module, "RUN_RWKV_6"):
        module.RUN_RWKV_6 = RUN_RWKV_6
    return module
