"""Carried states of infinite-context training (SURVEY.md 8 row a11): the same five names, constructor
arguments and indexing behaviour as src/infctx_module.py:3-50, so `src/model.py`'s infctx blocks
(`Block.forward(x, last_state: BlockState)`, :904-933) and `tmix_x060_forward(layer, x, last_state)`
take either implementation.

One extension: `BlockStateList.create/empty(..., wkv_dtype=torch.float32)` carries the WKV states in
fp32.  The reference stores them in bf16 whatever `dtype` says (src/infctx_module.py:36-38), i.e. it
rounds the state at every chunk boundary; `RUN_CUDA_RWKV6_STATE` accepts both.
"""
from dataclasses import dataclass

import torch


@dataclass
class TimeMixState:
    shift_state: torch.Tensor        # [B, C]            last token of the previous chunk (time-mix input)
    wkv_state: torch.Tensor          # [B, H, 64, 64]    WKV state, layout [value][key]


@dataclass
class ChannelMixState:
    shift_state: torch.Tensor        # [B, C]            last token of the previous chunk (channel-mix input)


@dataclass
class BlockState:
    time_mix_state: TimeMixState
    channel_mix_state: ChannelMixState


class BlockStateList:
    """All layers' states in two tensors: wkv_states [L, B, H, 64, 64], shift_states [L, 2, B, C]
    (index 0 = time mix, 1 = channel mix).  `states[layer]` returns views; `states[layer] = s` copies in."""

    def __init__(self, shift_states: torch.Tensor, wkv_states: torch.Tensor):
        self.wkv_states = wkv_states
        self.shift_states = shift_states

    @staticmethod
    def empty(N, B, C, H, device, dtype, wkv_dtype=torch.bfloat16):
        n = C // H
        return BlockStateList(torch.empty((N, 2, B, C), device=device, dtype=dtype),
                              torch.empty((N, B, H, n, n), device=device, dtype=wkv_dtype))

    @staticmethod
    def create(N, B, C, H, device, dtype, wkv_dtype=torch.bfloat16):
        out = BlockStateList.empty(N, B, C, H, device, dtype, wkv_dtype)
        out.wkv_states.zero_()
        out.shift_states.zero_()
        return out

    def __len__(self):
        return self.wkv_states.shape[0]

    def __getitem__(self, layer: int) -> BlockState:
        return BlockState(TimeMixState(self.shift_states[layer, 0], self.wkv_states[layer]),
                          ChannelMixState(self.shift_states[layer, 1]))

    def __setitem__(self, layer: int, state: BlockState):
        self.shift_states[layer, 0].copy_(state.time_mix_state.shift_state)
        self.wkv_states[layer].copy_(state.time_mix_state.wkv_state)
        self.shift_states[layer, 1].copy_(state.channel_mix_state.shift_state)

    def detach(self):
        """Truncated BPTT between chunks (the reference re-wraps `.detach()`ed tensors by hand)."""
        return BlockStateList(self.shift_states.detach(), self.wkv_states.detach())


# ------------------------------------------------------------------------------------------------
# whole-model training over a long sequence, one chunk of activations at a time
# ------------------------------------------------------------------------------------------------
def _shape_of(model):
    """(L, C, H) of a module tree with the reference's names (emb, blocks[i].att.time_faaaa)."""
    return len(model.blocks), model.emb.weight.shape[1], model.blocks[0].att.time_faaaa.shape[0]


def _check_states(model, states, B):
    L, C, H = _shape_of(model)
    if not isinstance(states, BlockStateList):
        raise TypeError(f"states must be a BlockStateList, got {type(states).__name__}")
    if tuple(states.wkv_states.shape) != (L, B, H, 64, 64):
        raise ValueError(f"states.wkv_states has shape {tuple(states.wkv_states.shape)}, the model needs {(L, B, H, 64, 64)}")
    if tuple(states.shift_states.shape) != (L, 2, B, C):
        raise ValueError(f"states.shift_states has shape {tuple(states.shift_states.shape)}, the model needs {(L, 2, B, C)}")
    if states.wkv_states.dtype not in (torch.bfloat16, torch.float32):
        raise ValueError(f"states.wkv_states must be bf16 or fp32, got {states.wkv_states.dtype}")


def _chunk_hidden(model, idx, wkv, att_shift, ffn_shift, exact):
    """ln_out(blocks(emb(idx))) of one chunk, starting from per-layer states (lists of L tensors: wkv [B,H,64,64],
    att_shift / ffn_shift [B,C]); returns (h, new wkv list, new att_shift list, new ffn_shift list).  The layers are
    those of encoders.blocks_forward (residual adds fused with the next LayerNorm), in the infctx flavour
    (src/model.py:869-902): the time mix takes (shift, wkv) and the channel mix its shift, and each returns its last
    input token as the next chunk's shift state."""
    from . import cmix, heads, tmix

    def ln(mod, x_, delta=None):
        return heads.add_layernorm(x_, delta, mod.weight, mod.bias, mod.eps)

    blocks = model.blocks
    n = len(blocks)
    fp32_gs = exact and wkv[0].dtype == torch.float32
    x, h = model.emb(idx), None
    new_wkv, new_att, new_ffn = [], [], []
    for i, blk in enumerate(blocks):
        if i == 0 and hasattr(blk, "ln0"):
            x = ln(blk.ln0, x)[1]
        if h is None:
            h = ln(blk.ln1, x)[1]
        a, (sa, sw) = tmix.tmix_x060_forward(blk.att, h, (att_shift[i], wkv[i]), exact_state_grad=exact,
                                             fp32_state_grad=fp32_gs)
        x, h = ln(blk.ln2, x, a)
        f, sf = cmix.cmix_x060_forward(blk.ffn, h, ffn_shift[i])
        x, h = ln(blocks[i + 1].ln1 if i + 1 < n else model.ln_out, x, f)
        new_wkv.append(sw)
        new_att.append(sa)
        new_ffn.append(sf)
    return h, new_wkv, new_att, new_ffn


def infctx_forward(model, idx, states, *, exact_state_grad=False):
    """One chunk of infctx training or inference (`RWKV.forward(idx, last_shift_states, last_wkv_states)`,
    src/model.py:1088-1132) on the fused kernels: (logits [B,T,vocab], new BlockStateList).

    `model` is any module tree with the reference's names: emb, blocks[i].{ln0 (i == 0), ln1, ln2, att, ffn}, ln_out,
    head (sft.RwkvSft, or the reference's own RWKV).  `states` is the BlockStateList the previous chunk returned (or
    `BlockStateList.create`).  The new states are new tensors (stacked, not copied into `states`), so they stay
    differentiable: with `exact_state_grad=True` the gradient of the new WKV states flows back into this chunk
    (ops.WKV_6STATE_BPTT; fp32 state gradients when the WKV states are fp32), otherwise the WKV state is a constant
    at the chunk boundary as in the reference.  The token-shift states are always differentiable."""
    L, C, H = _shape_of(model)
    _check_states(model, states, idx.shape[0])
    h, wkv, sa, sf = _chunk_hidden(model, idx, list(states.wkv_states.unbind(0)), list(states.shift_states[:, 0].unbind(0)),
                                   list(states.shift_states[:, 1].unbind(0)), exact_state_grad)
    shift = torch.stack([torch.stack(sa), torch.stack(sf)], 1)
    return model.head(h), BlockStateList(shift, torch.stack(wkv))


def infctx_train_step(model, idx, targets, chunk_ctx, *, exact=False, states=None, wkv_dtype=torch.float32):
    """Forward and backward of one long sequence, chunk by chunk, holding the activations of one chunk at a time.
    Returns (loss, final_states): the loss as a detached fp32 scalar and the detached BlockStateList after the last
    token.  Parameter gradients are accumulated into `.grad`; the caller zeroes them and steps the optimizer.

    idx, targets: int64 [B, T] (labels -100 are ignored).  The sequence is cut into chunks of `chunk_ctx` tokens (the
    last one may be shorter) and the loss is  sum_c (T_c / T) * sft_loss(logits_c, targets_c)  -- cross entropy plus
    L2Wrap per chunk (sft.sft_loss), so that with every label present the loss is the mean over the whole sequence.
    The reference's infctx `training_step` (src/model.py:1134-1192) sums per-chunk losses; its per-chunk weight has not
    been checked against the reference's source.  `states`: the initial BlockStateList (default zeros, WKV states in
    `wkv_dtype`).

    exact=False is the reference's truncated gradient: the WKV state is a constant at every chunk boundary
    (ops.WKV_6STATE_INFCTX), while the token-shift states are ordinary tensors whose gradient crosses it.
    exact=True also lets the WKV-state gradient cross the boundaries (ops.WKV_6STATE_BPTT, fp32 state gradients with
    the fp32 carry): the gradient of one pass over the whole sequence.

    Two sweeps.  The first runs the layers chunk by chunk and keeps only the states at every chunk start
    (L*B*H*16 KB + L*2*B*C*2 bytes per boundary with the fp32 carry).  The second walks the chunks in reverse: it
    recomputes a chunk from its stored starting states, made leaves that require grad, and back-propagates its loss
    together with the gradients the next chunk left on its starting states.  The first sweep runs with autograd
    enabled (one chunk's graph at a time, dropped at once, no head), so its WKV calls take the same time-segment plan
    as the recompute and the recomputed chunk reproduces the stored states bit for bit; a forward-only call may
    segment a chunk differently (DESIGN.md 4.4b).  Like torch.utils.checkpoint, the recompute of a chunk runs from the
    CPU and CUDA random-number states its first run started from, so dropout draws the same masks in both sweeps; the
    generators are left where one pass over the sequence leaves them."""
    if not isinstance(chunk_ctx, int) or chunk_ctx <= 0:
        raise ValueError(f"chunk_ctx must be a positive int, got {chunk_ctx!r}")
    if idx.dim() != 2 or tuple(targets.shape) != tuple(idx.shape):
        raise ValueError(f"idx and targets must both be [B, T], got {tuple(idx.shape)} and {tuple(targets.shape)}")
    B, T = idx.shape
    if T == 0:
        raise ValueError("idx has no tokens")
    L, C, H = _shape_of(model)
    dev = model.emb.weight.device
    if states is None:
        states = BlockStateList.create(L, B, C, H, dev, model.emb.weight.dtype, wkv_dtype=wkv_dtype)
    _check_states(model, states, B)
    from .sft import sft_loss

    bounds = [(t0, min(T, t0 + chunk_ctx)) for t0 in range(0, T, chunk_ctx)]

    def leaves(wkv, shift, grad_wkv):
        w = [s.detach().requires_grad_(grad_wkv) for s in wkv.unbind(0)]
        a = [s.detach().requires_grad_(True) for s in shift[:, 0].unbind(0)]
        f = [s.detach().requires_grad_(True) for s in shift[:, 1].unbind(0)]
        return w, a, f

    cuda = dev.type == "cuda"

    def rng_state():
        return torch.get_rng_state(), (torch.cuda.get_rng_state(dev) if cuda else None)

    def set_rng_state(st):
        torch.set_rng_state(st[0])
        if cuda:
            torch.cuda.set_rng_state(st[1], dev)

    # sweep 1: the states (and random-number states) at every chunk start; the last chunk's own final states come
    # from sweep 2
    starts = [(states.wkv_states.detach(), states.shift_states.detach())]
    rng = []
    with torch.enable_grad():
        for t0, t1 in bounds[:-1]:
            rng.append(rng_state())
            h, w, a, f = _chunk_hidden(model, idx[:, t0:t1], *leaves(*starts[-1], exact), exact)
            starts.append((torch.stack([s.detach() for s in w]),
                           torch.stack([torch.stack([s.detach() for s in a]), torch.stack([s.detach() for s in f])], 1)))
            del h, w, a, f                      # this chunk's graph goes before the next one is built
    rng.append(rng_state())
    # sweep 2: recompute each chunk with autograd, last chunk first
    total = torch.zeros((), dtype=torch.float32, device=dev)
    g_next, final = None, None
    with torch.enable_grad():
        for c in range(len(bounds) - 1, -1, -1):
            t0, t1 = bounds[c]
            w0, a0, f0 = leaves(*starts[c], exact)
            set_rng_state(rng[c])
            h, w, a, f = _chunk_hidden(model, idx[:, t0:t1], w0, a0, f0, exact)
            loss = sft_loss(model.head(h), targets[:, t0:t1]) * ((t1 - t0) / T)
            if final is None:
                rng_end = rng_state()
                final = BlockStateList(torch.stack([torch.stack([s.detach() for s in a]), torch.stack([s.detach() for s in f])], 1),
                                       torch.stack([s.detach() for s in w]))
            outs, grads = [loss], [None]
            if g_next is not None:
                for out_list, g_list in zip((w, a, f) if exact else (a, f), g_next):
                    for o, g in zip(out_list, g_list):
                        if g is not None:
                            outs.append(o)
                            grads.append(g)
            torch.autograd.backward(outs, grads)
            total += loss.detach().float()
            g_next = [[s.grad for s in lst] for lst in ((w0, a0, f0) if exact else (a0, f0))]
            del h, w, a, f, loss, outs, grads, w0, a0, f0
    set_rng_state(rng_end)
    return total, final
