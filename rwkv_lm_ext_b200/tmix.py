"""The whole RWKV-6 time-mix layer on the fused kernels (SURVEY.md section 8(f) rank 1).

`tmix_x060_forward(layer, x)` computes what `RWKV_Tmix_x060.forward` does (src/model.py:434-477):
token-shift + ddlerp, the five Linears (left to cuBLAS), the decay LoRA, WKV6, GroupNorm * gate and
the output Linear, on any module that carries the reference's parameter names

    time_maa_x/w/k/v/r/g [1,1,C]   time_maa_w1 [C,5R]   time_maa_w2 [5,R,C]
    time_decay [1,1,C]             time_decay_w1 [C,D]  time_decay_w2 [D,C]      time_faaaa [H,64]
    receptance, key, value, gate, output (bias-free Linears, plain or LoRA-wrapped)   ln_x (GroupNorm)

so it can be bound onto the reference's own layers without touching their state_dict:

    import types, rwkv_lm_ext_b200 as wkv
    for blk in model.blocks:
        blk.att.forward = types.MethodType(wkv.tmix_x060_forward, blk.att)

The eager chain's ~25 elementwise passes over [B,T,C] become 3 kernels (shift-lerp, ddlerp mix,
GroupNorm*gate) plus the `silu`; every piece is differentiable (heads.py, ops.py), so the same call
serves SFT.  Variants: `time_state` attribute present -> state tuning (src/model.py:560-584);
`last_state` given -> infctx (src/model.py:738-781): a `TimeMixState` (the reference's or
rwkv_lm_ext_b200.infctx's) returns `(out, TimeMixState(last_token, wkv_state))`, a plain
`(shift_state, wkv_state)` tuple returns `(out, (last_token, wkv_state))`.
With `exact_state_grad=True` the returned wkv_state is differentiable (ops.WKV_6STATE_BPTT): a model run chunk by
chunk over a long sequence, carrying both states, gets the gradients of one pass over the whole sequence.  The
default keeps the reference's truncated gradient, where the final wkv_state is a constant.
"""
import torch

from . import heads, ops


def _maa5(layer):
    C = layer.time_maa_w.shape[-1]
    ps = (layer.time_maa_w, layer.time_maa_k, layer.time_maa_v, layer.time_maa_r, layer.time_maa_g)
    if any(p.requires_grad for p in ps) and torch.is_grad_enabled():
        return torch.cat([p.view(1, C) for p in ps], 0)
    if ps[0].is_cuda and torch.cuda.is_current_stream_capturing():
        # inside a CUDA-graph capture the stacking has to be part of the graph: replays must read the live parameters
        return heads._bf16_param(torch.cat([p.detach().view(1, C) for p in ps], 0))
    # frozen (inference, LoRA SFT), eager: the stacked bf16 copy is kept until a parameter is written or moved
    key = tuple((p.data_ptr(), p._version, p.dtype) for p in ps)
    hit = layer.__dict__.get("_maa5_cache")
    if hit is None or hit[0] != key:
        with torch.no_grad():
            hit = (key, heads._bf16_param(torch.cat([p.detach().view(1, C) for p in ps], 0)))
        layer.__dict__["_maa5_cache"] = hit
    return hit[1]


def tmix_x060_project(layer, x, shift_state=None, gate_rows=None):
    """jit_func (src/model.py:434-459 / :738-762): x [B,T,C] bf16 -> r, k, v, g_raw, w (each [B,T,C]);
    g_raw is the gate Linear's output BEFORE silu (tmix_x060_finish applies it in-kernel).
    gate_rows: compute the gate for the first `gate_rows` batch rows only (the bidirectional encoders stack the reversed
    sequences behind the plain ones and never use their gate)."""
    B, T, C = x.shape
    bf = heads._bf16_param          # fp32 parameters (mixed-precision modules) are cast, never reinterpreted
    xxx = heads.tmix_shift_lerp(x, layer.time_maa_x, shift_state)
    h = torch.tanh(xxx.view(B * T, C) @ bf(layer.time_maa_w1))               # [B*T, 5R]
    xw, xk, xv, xr, xg = heads.tmix_ddlerp_lora(x, _maa5(layer), h, layer.time_maa_w2, shift_state)
    r = layer.receptance(xr)
    k = layer.key(xk)
    v = layer.value(xv)
    g = layer.gate(xg if gate_rows is None else xg[:gate_rows])      # raw: silu is applied inside the GroupNorm*gate kernel
    # time_decay + tanh(xw @ W1) @ W2 with the bias add as the GEMM epilogue
    w = torch.addmm(bf(layer.time_decay).view(-1), torch.tanh(xw.view(B * T, C) @ bf(layer.time_decay_w1)),
                    bf(layer.time_decay_w2)).view(B, T, -1)
    return r, k, v, g, w


def tmix_x060_finish(layer, y, g):
    """jit_func_2 (src/model.py:461-468): GroupNorm over heads, * silu(g_raw), output Linear."""
    H = layer.time_faaaa.shape[0]
    return layer.output(heads.groupnorm_gate(y, g, layer.ln_x.weight, layer.ln_x.bias, H, layer.ln_x.eps, gate_act="silu"))


def tmix_x060_forward(layer, x, last_state=None, *, exact_state_grad=False):
    """Drop-in for RWKV_Tmix_x060.forward (plain, state-tuning and infctx flavours).
    exact_state_grad (infctx only): let the gradient of the returned wkv_state flow back into this chunk."""
    B, T, C = x.shape
    H = layer.time_faaaa.shape[0]
    if last_state is not None:                                  # infctx: (shift_state [B,C], wkv_state [B,H,64,64])
        shift_state, wkv_state = (last_state.shift_state, last_state.wkv_state) if hasattr(last_state, "shift_state") else last_state
        r, k, v, g, w = tmix_x060_project(layer, x, shift_state)
        u = heads._bf16_param(layer.time_faaaa)
        if exact_state_grad:
            y, new_state = ops.WKV_6STATE_BPTT.apply(B, T, C, H, r, k, v, w, u, wkv_state.contiguous())
        else:
            y, new_state = ops.WKV_6STATE_INFCTX.apply(B, T, C, H, r, k, v, w, u, wkv_state.clone().contiguous())
        out = tmix_x060_finish(layer, y, g)
        if hasattr(last_state, "shift_state"):                  # reference calling convention (src/model.py:781)
            return out, type(last_state)(x[:, -1], new_state)
        return out, (x[:, -1], new_state)
    r, k, v, g, w = tmix_x060_project(layer, x)
    if getattr(layer, "time_state", None) is not None:          # state tuning
        y = ops.WKV_6STATE.apply(B, T, C, H, r, k, v, w, heads._bf16_param(layer.time_faaaa), heads._bf16_param(layer.time_state))
    else:
        y = ops.RUN_CUDA_RWKV6(B, T, C, H, r, k, v, w, heads._bf16_param(layer.time_faaaa))
    return tmix_x060_finish(layer, y, g)


class Tmix_x060(torch.nn.Module):
    """A self-contained layer with the reference's parameter names and initialisation shapes
    (src/model.py:375-432), for tests and benchmarks; real models keep their own layers and bind
    `tmix_x060_forward` onto them."""

    def __init__(self, n_embd, n_head, lora_r=32, decay_r=64, head_size_divisor=8, state_tuning=False):
        super().__init__()
        C = n_embd
        assert C == n_head * 64
        self.n_head = n_head
        z = lambda *s: torch.nn.Parameter(torch.zeros(*s))
        self.time_maa_x, self.time_maa_w, self.time_maa_k = z(1, 1, C), z(1, 1, C), z(1, 1, C)
        self.time_maa_v, self.time_maa_r, self.time_maa_g = z(1, 1, C), z(1, 1, C), z(1, 1, C)
        self.time_maa_w1, self.time_maa_w2 = z(C, 5 * lora_r), z(5, lora_r, C)
        self.time_decay, self.time_decay_w1, self.time_decay_w2 = z(1, 1, C), z(C, decay_r), z(decay_r, C)
        self.time_faaaa = z(n_head, 64)
        if state_tuning:
            self.time_state = z(n_head, 64, 64)
        self.receptance = torch.nn.Linear(C, C, bias=False)
        self.key = torch.nn.Linear(C, C, bias=False)
        self.value = torch.nn.Linear(C, C, bias=False)
        self.output = torch.nn.Linear(C, C, bias=False)
        self.gate = torch.nn.Linear(C, C, bias=False)
        self.ln_x = torch.nn.GroupNorm(n_head, C, eps=1e-5 * head_size_divisor ** 2)

    def forward(self, x, last_state=None, *, exact_state_grad=False):
        return tmix_x060_forward(self, x, last_state, exact_state_grad=exact_state_grad)
