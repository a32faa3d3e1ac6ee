"""Memory-bound pieces around the recurrence, with the reference's semantics:
eos / class-token gather (src/model_ext.py:209-211,1765), pooling (src/model_ext.py:1708-1738,
src/model_run.py:777-797), mask / reverse index / reverse gather (src/model_ext.py:398-419),
token-shift ddlerp (src/model.py:437-449) and GroupNorm*gate (src/model.py:461-467).
All arithmetic is in libwkv6_b200.so; these wrappers only allocate outputs."""
import torch

from . import _lib
from ._lib import check, ptr, stream_of


def _cuda(t):
    _lib.require_current_device(t)


def _dense(t):
    """t as a contiguous tensor whose data starts 16-byte aligned.  The kernels use 16-byte vector accesses and the
    library rejects a misaligned pointer, so a contiguous view at an element offset (`buf[1:].view(...)`) is copied
    into fresh storage first."""
    if t is None:
        return None
    t = t.contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


def _bf16_param(t):
    """Parameters reach the kernels as bf16.  A model kept in fp32 ('bf16-mixed', ln_x in fp32, ...) is cast here --
    differentiably, so the gradient returns in the parameter's own dtype -- instead of being reinterpreted."""
    if t is None:
        return None
    return _dense(t if t.dtype == torch.bfloat16 else t.to(torch.bfloat16))


def eos_index(idx: torch.Tensor, token_id: int) -> torch.Tensor:
    """== torch.eq(idx, token_id).int().argmax(-1): first occurrence, 0 if absent.  int64 [B]."""
    _cuda(idx)
    assert idx.dtype == torch.int64 and idx.dim() == 2
    idx = idx.contiguous()
    B, T = idx.shape
    pos = torch.empty(B, dtype=torch.int64, device=idx.device)
    check(_lib.load().eos_index_i64(B, T, ptr(idx), int(token_id), ptr(pos), stream_of(idx)), "eos_index_i64")
    return pos


def _ws(lib, B, T, C, nparam, device):
    return torch.empty(max(1, lib.elementwise_backward_workspace_bytes(B, T, C, nparam)), dtype=torch.uint8, device=device)


def _needs_grad(*ts):
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in ts)


def _gather_rows_fwd(x, pos):
    B, T, D = x.shape
    out = torch.empty(B, D, dtype=torch.bfloat16, device=x.device)
    check(_lib.load().gather_rows_bf16(B, T, D, ptr(x), ptr(pos), ptr(out), stream_of(x)), "gather_rows_bf16")
    return out


class _GatherRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, pos):
        ctx.save_for_backward(pos)
        ctx.shape = x.shape
        return _gather_rows_fwd(x, pos)

    @staticmethod
    def backward(ctx, gout):
        (pos,) = ctx.saved_tensors
        B, T, D = ctx.shape
        gout = _dense(gout)
        gx = torch.empty(B, T, D, dtype=torch.bfloat16, device=gout.device)
        check(_lib.load().scatter_rows_bf16(B, T, D, ptr(gout), ptr(pos), ptr(gx), stream_of(gout)), "scatter_rows_bf16")
        return gx, None


def gather_rows(x: torch.Tensor, pos: torch.Tensor) -> torch.Tensor:
    """== x[torch.arange(B), pos]  for x bf16 [B,T,D]  (differentiable w.r.t. x)."""
    _cuda(x)
    assert x.dtype == torch.bfloat16 and x.dim() == 3 and pos.dtype == torch.int64
    assert pos.numel() == x.shape[0], "one position per batch row"
    x, pos = _dense(x), pos.contiguous()
    if _needs_grad(x):
        assert x.shape[-1] % 8 == 0, "gather_rows under autograd needs D % 8 == 0 (scatter_rows_bf16)"
        return _GatherRows.apply(x, pos)
    return _gather_rows_fwd(x, pos)


def eos_gather(x: torch.Tensor, idx: torch.Tensor, token_id: int):
    """The classification / embedding head gather: (x[b, first eos], pos)."""
    pos = eos_index(idx, token_id)
    return gather_rows(x, pos), pos


_KIND = {"weightedmean": 0, "lasttoken": 1, "avg": 2}


def _pooling_fwd(x, alen, kind, variant):
    B, T, D = x.shape
    out = torch.empty(B, D, dtype=torch.float32, device=x.device)
    check(_lib.load().pooling_bf16(kind, variant, B, T, D, ptr(x), ptr(alen), ptr(out), stream_of(x)), "pooling_bf16")
    return out


class _Pooling(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, alen, kind, variant):
        ctx.save_for_backward(alen)
        ctx.meta = (x.shape, kind, variant)
        return _pooling_fwd(x, alen, kind, variant)

    @staticmethod
    def backward(ctx, gout):
        (alen,) = ctx.saved_tensors
        (B, T, D), kind, variant = ctx.meta
        gout = _dense(gout.float())
        gx = torch.empty(B, T, D, dtype=torch.bfloat16, device=gout.device)
        check(_lib.load().pooling_backward_bf16(kind, variant, B, T, D, ptr(alen), ptr(gout), ptr(gx), stream_of(gout)),
              "pooling_backward_bf16")
        return gx, None, None, None


def pooling(x: torch.Tensor, actual_len: torch.Tensor, pooling_type: str, variant: str = "train") -> torch.Tensor:
    """variant="train": src/model_ext.py:1708-1738 (bf16 result for weightedmean / avg);
    variant="infer": src/model_run.py:777-797 (L = actual_len + 1, fp32 result).
    Differentiable w.r.t. x."""
    _cuda(x)
    assert x.dtype == torch.bfloat16 and x.dim() == 3
    if pooling_type == "lasttoken":
        return gather_rows(x, actual_len.to(torch.int64))
    if pooling_type not in _KIND or (variant == "infer" and pooling_type == "avg"):
        raise ValueError(pooling_type)
    x = _dense(x)
    alen = actual_len.to(torch.int64).contiguous()
    kind, var = _KIND[pooling_type], 1 if variant == "infer" else 0
    out = _Pooling.apply(x, alen, kind, var) if _needs_grad(x) else _pooling_fwd(x, alen, kind, var)
    return out.bfloat16() if variant == "train" else out


def create_mask_and_rev_idx(idx: torch.Tensor, emb_id: int = 1, pad_id: int = 0):
    """create_mask + reverse_x_idx (src/model_ext.py:398-417) in one launch, on the device
    (the reference builds rev_idx with a Python loop over the batch on the host)."""
    _cuda(idx)
    assert idx.dtype == torch.int64 and idx.dim() == 2
    idx = idx.contiguous()
    B, T = idx.shape
    mask = torch.empty(B, T, dtype=torch.int32, device=idx.device)
    rev = torch.empty(B, T, dtype=torch.int64, device=idx.device)
    check(_lib.load().create_mask_rev_idx(B, T, ptr(idx), int(emb_id), int(pad_id), ptr(mask), ptr(rev), stream_of(idx)),
          "create_mask_rev_idx")
    return mask, rev


def _reverse_fwd(x, rev_idx):
    B, T, D = x.shape
    out = torch.empty_like(x)
    check(_lib.load().gather_tokens_bf16(B, T, D, ptr(x), ptr(rev_idx), ptr(out), stream_of(x)), "gather_tokens_bf16")
    return out


class _ReverseX(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, rev_idx):
        ctx.save_for_backward(rev_idx)
        return _reverse_fwd(x, rev_idx)

    @staticmethod
    def backward(ctx, gout):
        (rev_idx,) = ctx.saved_tensors
        gout = _dense(gout)
        B, T, D = gout.shape
        gx = torch.empty_like(gout)
        check(_lib.load().scatter_tokens_bf16(B, T, D, ptr(gout), ptr(rev_idx), ptr(gx), stream_of(gout)), "scatter_tokens_bf16")
        return gx, None


def stack_reversed(x: torch.Tensor, rev_idx: torch.Tensor) -> torch.Tensor:
    """cat([x, reverse_x(x, rev_idx)], 0)  [2B,T,D]: both directions of a bidirectional encoder layer as one batch.
    One kernel (x read once) when no gradient is needed; the differentiable pieces otherwise."""
    _cuda(x)
    if _needs_grad(x) or x.shape[-1] % 8 != 0:
        return torch.cat([x, reverse_x(x, rev_idx)], 0)
    assert x.dtype == torch.bfloat16 and x.dim() == 3 and rev_idx.dtype == torch.int64 and rev_idx.shape == x.shape[:2]
    x, rev_idx = _dense(x), rev_idx.contiguous()
    B, T, D = x.shape
    out = torch.empty((2 * B, T, D), device=x.device, dtype=x.dtype)
    check(_lib.load().stack_reversed_bf16(B, T, D, ptr(x), ptr(rev_idx), ptr(out), stream_of(x)), "stack_reversed_bf16")
    return out


def reverse_x(x: torch.Tensor, rev_idx: torch.Tensor) -> torch.Tensor:
    """== torch.gather(x, 1, rev_idx[..., None].expand(-1, -1, D))  (src/model_ext.py:418-419).
    Differentiable w.r.t. x when rev_idx is a per-row permutation (what reverse_x_idx builds)."""
    _cuda(x)
    assert x.dtype == torch.bfloat16 and x.dim() == 3 and rev_idx.dtype == torch.int64
    x, rev_idx = _dense(x), rev_idx.contiguous()
    if _needs_grad(x):
        return _ReverseX.apply(x, rev_idx)
    return _reverse_fwd(x, rev_idx)


def _shift_lerp_fwd(x, shift_state, maa_x):
    B, T, C = x.shape
    out = torch.empty_like(x)
    check(_lib.load().tmix_shift_lerp_bf16(B, T, C, ptr(x), ptr(shift_state), ptr(maa_x), ptr(out), stream_of(x)),
          "tmix_shift_lerp_bf16")
    return out


class _ShiftLerp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, shift_state, maa_x):
        ctx.save_for_backward(x, shift_state, maa_x)
        return _shift_lerp_fwd(x, shift_state, maa_x)

    @staticmethod
    def backward(ctx, gout):
        x, shift_state, maa_x = ctx.saved_tensors
        lib = _lib.load()
        B, T, C = x.shape
        gout = _dense(gout)
        gx = torch.empty_like(x)
        gmaa = torch.empty(C, dtype=torch.float32, device=x.device) if ctx.needs_input_grad[2] else None   # frozen: no reduction
        gshift = torch.empty_like(shift_state) if shift_state is not None else None
        ws = _ws(lib, B, T, C, 1, x.device)
        check(lib.tmix_shift_lerp_backward_bf16(B, T, C, ptr(x), ptr(shift_state), ptr(maa_x), ptr(gout), ptr(gx), ptr(gmaa),
                                                ptr(gshift), ptr(ws), ws.numel(), stream_of(x)), "tmix_shift_lerp_backward_bf16")
        return gx, gshift, (gmaa.to(maa_x.dtype) if gmaa is not None else None)


def tmix_shift_lerp(x, maa_x, shift_state=None):
    """xxx = x + (time_shift(x) - x) * time_maa_x  (src/model.py:437-439).  Differentiable w.r.t.
    x, time_maa_x and the shift state."""
    _cuda(x)
    assert x.dtype == torch.bfloat16
    x = _dense(x)
    flat = _bf16_param(maa_x).view(-1)
    assert flat.numel() == x.shape[-1]
    shift_state = _bf16_param(shift_state)
    if _needs_grad(x, maa_x, shift_state):
        return _ShiftLerp.apply(x, shift_state, flat)
    return _shift_lerp_fwd(x, shift_state, flat)


def _ddlerp_fwd(x, shift_state, maa, m):
    B, T, C = x.shape
    out = torch.empty(5, B, T, C, dtype=torch.bfloat16, device=x.device)
    check(_lib.load().tmix_ddlerp_mix_bf16(B, T, C, ptr(x), ptr(shift_state), ptr(maa), ptr(m), ptr(out), stream_of(x)),
          "tmix_ddlerp_mix_bf16")
    return out


def _ddlerp_bwd(x, shift_state, maa, m, gouts, need_gmaa):
    """(gx, gshift, gmaa, gm) of x + xx * (maa_n + m_n) for the five incoming gradients (None = zero)"""
    lib = _lib.load()
    B, T, C = x.shape
    gouts = [torch.zeros_like(x) if g is None else _dense(g) for g in gouts]
    gx, gm = torch.empty_like(x), torch.empty_like(m)
    gmaa = torch.empty(5, C, dtype=torch.float32, device=x.device) if need_gmaa else None
    gshift = torch.empty_like(shift_state) if shift_state is not None else None
    ws = _ws(lib, B, T, C, 5, x.device)
    check(lib.tmix_ddlerp_mix_backward_bf16(B, T, C, ptr(x), ptr(shift_state), ptr(maa), ptr(m), *[ptr(g) for g in gouts],
                                            ptr(gx), ptr(gm), ptr(gmaa), ptr(gshift), ptr(ws), ws.numel(), stream_of(x)),
          "tmix_ddlerp_mix_backward_bf16")
    return gx, gshift, (gmaa.to(maa.dtype) if gmaa is not None else None), gm


class _DdlerpMix(torch.autograd.Function):
    """Five outputs (views of one [5,B,T,C] buffer), five incoming gradients: the consumers are five
    different Linears, so autograd never has to stack their gradients into one tensor."""

    @staticmethod
    def forward(ctx, x, shift_state, maa, m):
        ctx.save_for_backward(x, shift_state, maa, m)
        return tuple(_ddlerp_fwd(x, shift_state, maa, m).unbind(0))

    @staticmethod
    def backward(ctx, *gouts):
        x, shift_state, maa, m = ctx.saved_tensors
        return _ddlerp_bwd(x, shift_state, maa, m, gouts, ctx.needs_input_grad[2])


def tmix_ddlerp_mix(x, maa_wkvrg, m, shift_state=None):
    """xw,xk,xv,xr,xg = x + xx * (time_maa_n + m_n)  (src/model.py:444-448).
    maa_wkvrg bf16 [5,C]; m bf16 [5,B,T,C] (the LoRA bmm output).  Returns a [5,B,T,C] tensor
    (inference) or the tuple of its five [B,T,C] slices (when a gradient is needed): unpack or index
    it either way.  Differentiable w.r.t. x, maa_wkvrg, m and the shift state."""
    _cuda(x)
    assert x.dtype == torch.bfloat16 and m.dtype == torch.bfloat16
    x, m, maa = _dense(x), _dense(m), _bf16_param(maa_wkvrg)
    assert tuple(maa.shape) == (5, x.shape[-1]) and tuple(m.shape) == (5,) + tuple(x.shape)
    shift_state = _bf16_param(shift_state)
    if _needs_grad(x, maa, m, shift_state):
        return _DdlerpMix.apply(x, shift_state, maa, m)
    return _ddlerp_fwd(x, shift_state, maa, m)


class _DdlerpLora(torch.autograd.Function):
    """Forward: the fused kernel (m never leaves the chip).  Backward: m is recomputed with one bmm, the
    TMA-fed ddlerp backward gives gx / gm / gmaa, two more bmm carry gm to h and W2."""

    @staticmethod
    def forward(ctx, x, shift_state, maa, h, w2):
        ctx.save_for_backward(x, shift_state, maa, h, w2)
        return tuple(_ddlerp_lora_fwd(x, shift_state, maa, h, w2).unbind(0))

    @staticmethod
    def backward(ctx, *gouts):
        x, shift_state, maa, h, w2 = ctx.saved_tensors
        B, T, C = x.shape
        R = w2.shape[1]
        h5 = h.view(B * T, 5, R).transpose(0, 1)                     # [5, BT, R]
        m = torch.bmm(h5, w2).view(5, B, T, C)
        need = ctx.needs_input_grad                                  # frozen parameters (LoRA SFT): no cast, no bmm
        gx, gshift, gmaa, gm = _ddlerp_bwd(x, shift_state, maa, m, gouts, need[2])
        gm5 = gm.view(5, B * T, C)
        gh = torch.bmm(gm5, w2.transpose(1, 2)).transpose(0, 1).reshape(B * T, 5 * R).view_as(h) if need[3] else None
        gw2 = torch.bmm(h5.transpose(1, 2), gm5) if need[4] else None
        return gx, gshift, gmaa, gh, gw2


def _ddlerp_lora_fwd(x, shift_state, maa, h, w2):
    B, T, C = x.shape
    out = torch.empty(5, B, T, C, dtype=torch.bfloat16, device=x.device)
    check(_lib.load().tmix_ddlerp_lora_bf16(B, T, C, w2.shape[1], ptr(x), ptr(shift_state), ptr(maa), ptr(h), ptr(w2), ptr(out),
                                            stream_of(x)), "tmix_ddlerp_lora_bf16")
    return out


def tmix_ddlerp_lora(x, maa_wkvrg, h, w2, shift_state=None):
    """xw,xk,xv,xr,xg = x + xx * (time_maa_n + h_n @ W2_n)  (src/model.py:442-448) with the rank-R LoRA
    product on the tensor cores inside the kernel.  h bf16 [B*T, 5R] or [B,T,5R] = tanh(xxx @ W1);
    w2 bf16 [5,R,C].  R = 32 and C % 64 == 0; other shapes take the bmm + tmix_ddlerp_mix route.
    Returns five [B,T,C] tensors (a tuple under autograd, a [5,B,T,C] tensor otherwise)."""
    _cuda(x)
    assert x.dtype == torch.bfloat16 and h.dtype == torch.bfloat16
    B, T, C = x.shape
    R = w2.shape[1]
    x, maa, w2 = _dense(x), _bf16_param(maa_wkvrg), _bf16_param(w2)
    assert tuple(maa.shape) == (5, C) and tuple(w2.shape) == (5, R, C)
    h = _dense(h).view(B * T, 5 * R)
    shift_state = _bf16_param(shift_state)
    if R != 32 or C % 64 != 0:
        m = torch.bmm(h.view(B * T, 5, R).transpose(0, 1), w2).view(5, B, T, C)
        return tmix_ddlerp_mix(x, maa, m, shift_state)
    if _needs_grad(x, maa, h, w2, shift_state):
        return _DdlerpLora.apply(x, shift_state, maa, h, w2)
    return _ddlerp_lora_fwd(x, shift_state, maa, h, w2)


_GATE_ACT = {None: 0, "none": 0, "silu": 1}


def _gn_fwd(y, g, ln_w, ln_b, H, eps, act):
    B, T, C = y.shape
    out = torch.empty_like(y)
    check(_lib.load().groupnorm_gate_bf16(B * T, C, H, float(eps), act, ptr(y), ptr(g), ptr(ln_w), ptr(ln_b), ptr(out),
                                          stream_of(y)), "groupnorm_gate_bf16")
    return out


class _GroupNormGate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, y, g, ln_w, ln_b, H, eps, act):
        ctx.save_for_backward(y, g, ln_w, ln_b)
        ctx.meta = (H, eps, act)
        return _gn_fwd(y, g, ln_w, ln_b, H, eps, act)

    @staticmethod
    def backward(ctx, gout):
        y, g, ln_w, ln_b = ctx.saved_tensors
        H, eps, act = ctx.meta
        lib = _lib.load()
        B, T, C = y.shape
        gout = _dense(gout)
        gy, gg = torch.empty_like(y), torch.empty_like(g)
        need_p = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]                       # frozen affine: no reduction
        gw = torch.empty(C, dtype=torch.float32, device=y.device) if need_p else None
        gb = torch.empty(C, dtype=torch.float32, device=y.device) if need_p else None
        ws = _ws(lib, B, T, C, 2, y.device)
        check(lib.groupnorm_gate_backward_bf16(B * T, C, H, float(eps), act, ptr(y), ptr(g), ptr(ln_w), ptr(ln_b), ptr(gout),
                                               ptr(gy), ptr(gg), ptr(gw), ptr(gb), ptr(ws), ws.numel(), stream_of(y)),
              "groupnorm_gate_backward_bf16")
        return gy, gg, (gw.to(ln_w.dtype) if need_p else None), (gb.to(ln_b.dtype) if need_p else None), None, None, None


def groupnorm_gate(y, g, ln_w, ln_b, H, eps, gate_act=None):
    """ln_x(y.view(B*T, C)).view(B,T,C) * g  (src/model.py:461-467, without the output Linear).
    gate_act="silu": g is the gate Linear's raw output and F.silu (src/model.py:454) is applied
    inside the kernel.  Differentiable w.r.t. y, g and the GroupNorm affine parameters."""
    _cuda(y)
    assert y.dtype == torch.bfloat16 and g.dtype == torch.bfloat16
    y, g, ln_w, ln_b = _dense(y), _dense(g), _bf16_param(ln_w), _bf16_param(ln_b)
    assert ln_w.numel() == y.shape[-1] and ln_b.numel() == y.shape[-1] and y.shape[-1] == H * 64
    act = _GATE_ACT[gate_act]
    if _needs_grad(y, g, ln_w, ln_b):
        return _GroupNormGate.apply(y, g, ln_w, ln_b, H, eps, act)
    return _gn_fwd(y, g, ln_w, ln_b, H, eps, act)


def groupnorm_gate_pair(y, y_rev, rev_idx, g, ln_w, ln_b, H, eps, gate_act=None):
    """ln_x((y + reverse_x(y_rev, rev_idx)) / 2) * g  -- the tail of bi_att_forward_batch
    (src/model_encoder_run.py:72-74) with the reverse gather and the average inside the kernel.
    Under autograd the pieces run separately (each is differentiable)."""
    _cuda(y)
    if _needs_grad(y, y_rev, g, ln_w, ln_b):
        return groupnorm_gate((y + reverse_x(y_rev, rev_idx)) / 2, g, ln_w, ln_b, H, eps, gate_act)
    assert y.dtype == torch.bfloat16 and y_rev.dtype == torch.bfloat16 and g.dtype == torch.bfloat16 and rev_idx.dtype == torch.int64
    y, y_rev, g, rev_idx = _dense(y), _dense(y_rev), _dense(g), rev_idx.contiguous()
    B, T, C = y.shape
    out = torch.empty_like(y)
    check(_lib.load().groupnorm_gate_pair_bf16(B, T, C, H, float(eps), _GATE_ACT[gate_act], ptr(y), ptr(y_rev), ptr(rev_idx), ptr(g),
                                               ptr(_bf16_param(ln_w)), ptr(_bf16_param(ln_b)), ptr(out), stream_of(y)),
          "groupnorm_gate_pair_bf16")
    return out


def _add_ln_fwd(x, delta, w, b, eps, want_stats):
    D = x.shape[-1]
    rows = x.numel() // D
    y = torch.empty_like(x)
    x_new = torch.empty_like(x) if delta is not None else None
    stats = torch.empty(rows, 2, dtype=torch.float32, device=x.device) if want_stats else None
    check(_lib.load().add_layernorm_bf16(rows, D, float(eps), ptr(x), ptr(delta), ptr(w), ptr(b), ptr(x_new), ptr(y),
                                         ptr(stats), stream_of(x)), "add_layernorm_bf16")
    return (x if delta is None else x_new), y, stats


def _add_ln_bwd(ctx, g_xnew, g_y):
    x_new, stats, w = ctx.saved_tensors
    lib = _lib.load()
    D = x_new.shape[-1]
    rows = x_new.numel() // D
    if g_y is None:                              # only the residual stream carried a gradient
        return g_xnew, None, None
    g_y = g_y.contiguous()
    g_xnew = g_xnew.contiguous() if g_xnew is not None else None
    g = torch.empty_like(x_new)
    need_p = ctx.needs_input_grad[ctx.w_index] or ctx.needs_input_grad[ctx.w_index + 1]
    gw = torch.empty(D, dtype=torch.float32, device=x_new.device) if need_p else None
    gb = torch.empty(D, dtype=torch.float32, device=x_new.device) if need_p else None
    n = lib.add_layernorm_backward_workspace_bytes(rows, D) if need_p else 0
    ws = torch.empty(max(n, 1), dtype=torch.uint8, device=x_new.device) if need_p else None
    check(lib.add_layernorm_backward_bf16(rows, D, ptr(x_new), ptr(stats), ptr(w), ptr(g_y), ptr(g_xnew), ptr(g), ptr(gw),
                                          ptr(gb), ptr(ws), n, stream_of(x_new)), "add_layernorm_backward_bf16")
    return g, (gw.to(w.dtype) if need_p else None), (gb.to(w.dtype) if need_p else None)


class _AddLayerNorm(torch.autograd.Function):
    """(x, delta) -> (x + delta, LayerNorm(x + delta)); one gradient tensor serves x and delta."""

    @staticmethod
    def forward(ctx, x, delta, w, b, eps):
        x_new, y, stats = _add_ln_fwd(x, delta, w, b, eps, True)
        ctx.save_for_backward(x_new, stats, w)
        ctx.w_index = 2
        return x_new, y

    @staticmethod
    def backward(ctx, g_xnew, g_y):
        g, gw, gb = _add_ln_bwd(ctx, g_xnew, g_y)
        return g, g, gw, gb, None


class _LayerNorm(torch.autograd.Function):
    """x -> LayerNorm(x) on the same kernels (no residual operand)."""

    @staticmethod
    def forward(ctx, x, w, b, eps):
        _, y, stats = _add_ln_fwd(x, None, w, b, eps, True)
        ctx.save_for_backward(x, stats, w)
        ctx.w_index = 1
        return y

    @staticmethod
    def backward(ctx, g_y):
        g, gw, gb = _add_ln_bwd(ctx, None, g_y)
        return g, gw, gb, None


def add_layernorm(x, delta, ln_w, ln_b, eps=1e-5):
    """(x_new, y) with x_new = x + delta and y = LayerNorm(x_new) -- the residual add and the next LayerNorm of
    `Block.forward` (src/model.py:904-933) in one pass over the residual stream.  delta = None: y = LayerNorm(x),
    x_new is x.  bf16 [..., D], D % 256 == 0 (other widths take the eager route).  Differentiable w.r.t. x, delta
    and the affine parameters (their column pass is skipped when they are frozen)."""
    _cuda(x)
    assert x.dtype == torch.bfloat16
    D = x.shape[-1]
    if D % 256 != 0:
        x_new = x if delta is None else x + delta
        return x_new, torch.nn.functional.layer_norm(x_new, (D,), ln_w, ln_b, eps)
    x = x.contiguous()
    delta = delta.contiguous() if delta is not None else None
    w, b = _bf16_param(ln_w), _bf16_param(ln_b)
    if _needs_grad(x, delta, w, b):
        if delta is None:
            return x, _LayerNorm.apply(x, w, b, eps)
        return _AddLayerNorm.apply(x, delta, w, b, eps)
    x_new, y, _ = _add_ln_fwd(x, delta, w, b, eps, False)
    return x_new, y
