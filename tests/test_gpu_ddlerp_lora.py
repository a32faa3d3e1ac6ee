"""The fused LoRA ddlerp forward (csrc/ddlerp_lora.cu through heads.tmix_ddlerp_lora) at the pipeline depths the models
run, every output element against the bf16 chain of the exact LoRA product; its bmm route for other ranks; its
backward at a model shape.  `pytest -m gpu`.

A CTA takes 128 token rows and `gpc` consecutive 64-channel groups: 5 * gpc work items (group, output).  The x tile of a
group is double-buffered and refilled once the epilogue has finished the group two back, the W2 tiles go through a
ring of three slots, the accumulators alternate between two TMEM buffers.  The host picks gpc from the shape
(ddlerp_lora_forward, restated by `plan` below):

    shape (B*T, C)                who runs it                               gpc        last CTA   items per CTA
    74,256 / 390,768 / 600,2048   test_ddlerp_lora_fused                    2 / 2 / 2  2 / 2 / 2  <= 10
    1, 64                         test_ddlerp_lora_fused                    1          1          5
    231, 320                      test_no_writes_outside_the_outputs        3          2          15
    600, 448                      here                                      3          1          15
    32768, 2048                   1B6 training, 8 x 4096                    7          4          35
    65536, 2048                   bi-encoder, 64 passages x 2 dirs x 512    11         10         55
    65536, 2560                   3B, 16 x 4096                             14         12         70
    32768, 4096                   7B shape, 8 x 4096, at rank 32            13         12         65

(last CTA: the groups of the grid's last channel split.)

Only grids with gpc >= 3 refill an x buffer, and only the model shapes take the W2 ring and the accumulator barriers
through dozens of phases or end a CTA on fewer groups than gpc.

The contract.  The epilogue does the reference's bf16 operations one by one,

    out_n = x + xx * (maa_n + bf16(m_n)),   xx = shift(x) - x,   m_n = h_n @ W2_n  (K = 32, fp32 accumulation),

so each output is fixed once the bf16 value of m is.  m64 (fp64, exact: the bf16 products are exact and 32 of them
sum without loss) and s64 = |h_n| @ |W2_n| bound where the kernel's fp32 sum can land: within delta = 2^-20 * s64 of
m64.  That is 16 fp32 roundings of 2^-24 * s64 each; a tree-ordered sum of 32 products rounds 5 times along any path,
a sequential one up to 31 times, and the tensor cores' internal accumulation precision is not documented, so the
margin is what the test relies on (no element has fallen outside it at the shapes below).  Rounding to bf16 and every
step of the chain are monotone in m (round-to-nearest additions, a multiplication by a fixed xx), so every output must
lie between chain(lo) and chain(hi), lo / hi the bf16 values just below m64 - delta / just above m64 + delta.  That
holds whatever order the tensor cores sum in, and a wrong row, group, plane, W2 slot or stale x buffer breaks it.
Without delta, rows where the sum cancels would fail: there the bf16 spacing at m is finer than the accumulation error.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"
R = 32
DELTA = 2.0 ** -20
# share of outputs allowed to differ from chain(RN(m64)), where the fp32 sum flipped a bf16 rounding of m: measured at
# most 2.3e-6 per shape here (about 1e-6 at the model shapes) on a B200 at its 1000 W power limit
MAX_OFF_CHAIN = 0.01


@pytest.fixture(scope="module")
def M():
    import rwkv_lm_ext_b200 as M
    M.load()
    return M


def plan(BT, C):
    """(tiles, split, gpc, groups of the last CTA) as ddlerp_lora_forward chooses them: about four waves of CTAs
    (2 resident on each of 148 SMs), at least two groups per CTA where there are two"""
    tiles, groups = -(-BT // 128), C // 64
    split = (148 * 2 * 4 + tiles - 1) // tiles
    split = max(min(split, groups // 2), 1)
    gpc = -(-groups // split)
    split = -(-groups // gpc)
    return tiles, split, gpc, groups - (split - 1) * gpc


def _inputs(B, T, C, with_state, seed, rank=R):
    """device-side generators, the magnitudes of test_ddlerp_lora_fused"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    x = torch.randn(B, T, C, generator=g, device=DEV).bfloat16()
    maa = torch.rand(5, C, generator=g, device=DEV).bfloat16()
    h = torch.tanh(torch.randn(B * T, 5 * rank, generator=g, device=DEV)).bfloat16()
    w2 = (torch.randn(5, rank, C, generator=g, device=DEV) * 0.1).bfloat16()
    st = torch.randn(B, C, generator=g, device=DEV).bfloat16() if with_state else None
    return x, maa, h, w2, st


# ------------------------------------------------------------------------------------------------------------------
# the element-wise contract
# ------------------------------------------------------------------------------------------------------------------
def _bf16_step(b, up):
    """the bf16 neighbour of every (finite) element of b, above it (up) or below it, by stepping its bit pattern"""
    u = b.view(torch.int16).to(torch.int32) & 0xFFFF
    sign, mag = u >> 15, u & 0x7FFF
    step = 1 if up else -1
    mag2 = mag + torch.where(sign == 0, step, -step)       # a positive value moves with the step, a negative one against it
    zero = mag == 0                                        # +-0 steps to the smallest subnormal of the step's sign
    sign2 = torch.where(zero, torch.full_like(sign, 0 if up else 1), sign)
    bits = (sign2 << 15) | torch.where(zero, torch.ones_like(mag2), mag2)
    return (bits - ((bits >> 15) << 16)).to(torch.int16).view(torch.bfloat16)


def _bf16_below(v):
    """the largest bf16 value <= v (fp64).  v.to(bf16) is one of the two bf16 neighbours of v however torch rounds
    (fp64 -> fp32 -> bf16 rounds twice); the comparison in fp64 picks the lower one."""
    r = v.to(torch.bfloat16)
    return torch.where(r.double() > v, _bf16_step(r, up=False), r)


def _bf16_above(v):
    r = v.to(torch.bfloat16)
    return torch.where(r.double() < v, _bf16_step(r, up=True), r)


def _bf16_nearest(v):
    """round-to-nearest-even of fp64 v to bf16, in one rounding"""
    lo, hi = _bf16_below(v), _bf16_above(v)
    dlo, dhi = v - lo.double(), hi.double() - v
    hi_even = (hi.view(torch.int16) & 1) == 0
    return torch.where((dhi < dlo) | ((dhi == dlo) & hi_even), hi, lo)


def _eager_shift(x, st):
    """the reference's bf16 xx = shift(x) - x (nn.ZeroPad2d((0,0,1,-1)), or the infctx shift state at t == 0)"""
    prev = torch.zeros_like(x[:, :1]) if st is None else st.unsqueeze(1)
    return torch.cat([prev, x[:, :-1]], 1) - x


def _chain(x, xx, maa_n, m):
    """src/model.py:444-448 as torch bf16 operations, bit-equal to tmix_ddlerp_mix (test_ddlerp_matches_eager_bf16_chain)"""
    return x + xx * (maa_n + m)


def assert_ddlerp_contract(out, x, maa, h, w2, st, what):
    """every element of the five [B,T,C] planes of out within [chain(lo), chain(hi)] (module docstring); returns the
    share of elements that differ from chain(RN(m64))"""
    B, T, C = x.shape
    rank = w2.shape[1]
    xx = _eager_shift(x, st)
    h5 = h.view(B * T, 5, rank)
    off = 0
    for n in range(5):                                     # one plane at a time bounds the fp64 temporaries
        hn, wn = h5[:, n].double(), w2[n].double()
        m64 = (hn @ wn).view(B, T, C)
        d = (hn.abs() @ wn.abs()).view(B, T, C) * DELTA
        c_lo = _chain(x, xx, maa[n], _bf16_below(m64 - d))
        c_hi = _chain(x, xx, maa[n], _bf16_above(m64 + d))
        got = out[n]
        ok = (got >= torch.minimum(c_lo, c_hi)) & (got <= torch.maximum(c_lo, c_hi))      # NaN fails too
        if not bool(ok.all()):
            bad = (~ok).nonzero()
            b, t, c = bad[0].tolist()
            row = b * T + t
            raise AssertionError(
                f"{what}: output {n}: {bad.shape[0]} of {got.numel()} elements outside [chain(lo), chain(hi)]; first at "
                f"b={b} t={t} c={c} (tile {row // 128}, tile row {row % 128}, group {c // 64}): got {got[b, t, c].item()}, "
                f"chain(lo) {c_lo[b, t, c].item()}, chain(hi) {c_hi[b, t, c].item()}, m64 {m64[b, t, c].item():.6g}, "
                f"x {x[b, t, c].item()}, xx {xx[b, t, c].item()}, maa {maa[n, c].item()}")
        off += int((got != _chain(x, xx, maa[n], _bf16_nearest(m64))).sum())
    return off / out.numel()


# ------------------------------------------------------------------------------------------------------------------
# forward: the contract at every pipeline depth
# ------------------------------------------------------------------------------------------------------------------
# (B, T, C, with_state, gpc, groups of the last CTA)
SHAPES = [
    (2, 37, 256, False, 2, 2), (2, 37, 256, True, 2, 2),          # the shapes of test_ddlerp_lora_fused
    (3, 130, 768, False, 2, 2), (3, 130, 768, True, 2, 2),
    (1, 1, 64, False, 1, 1), (1, 1, 64, True, 1, 1),
    (2, 300, 2048, False, 2, 2), (2, 300, 2048, True, 2, 2),
    (2, 300, 448, True, 3, 1),            # a last CTA of one group (ngroups == 1) in a multi-CTA grid
    (8, 4096, 2048, False, 7, 4),         # 1B6 training: batch starts at tile row 0
    (13, 2521, 2048, True, 7, 4),         # ... and at other rows, 5 live rows in the last tile
    (128, 512, 2048, True, 11, 10),       # bi-encoder, both directions stacked
    (508, 129, 2048, False, 11, 10),      # T = 129: each tile has its batch start at another row
    (16, 4096, 2560, True, 14, 12),       # 3B
    (500, 131, 2560, False, 14, 12),
    (8, 4096, 4096, False, 13, 12),       # 7B shape at rank 32
    # T = 1: every row is t == 0 and reads its own row of the shift state from global memory at the start of each group,
    # which slows the epilogue against the issuer; a release of the x buffer ahead of its reads showed here
    (32768, 1, 4096, True, 13, 12),
]


@pytest.mark.parametrize("B,T,C,with_state,gpc,last", SHAPES,
                         ids=[f"{B}x{T}x{C}{'_state' if s else ''}" for B, T, C, s, _, _ in SHAPES])
def test_forward_within_the_bf16_chain_of_the_exact_product(M, B, T, C, with_state, gpc, last):
    assert plan(B * T, C)[2:] == (gpc, last), plan(B * T, C)
    x, maa, h, w2, st = _inputs(B, T, C, with_state, seed=B * T + C)
    out = M.tmix_ddlerp_lora(x, maa, h, w2, st)
    assert out.shape == (5, B, T, C)
    frac = assert_ddlerp_contract(out, x, maa, h, w2, st, f"{B}x{T}x{C}")
    print(f"ddlerp_lora {B}x{T}x{C}{' state' if with_state else ''}: {frac:.3e} of the outputs differ from chain(RN(m64))")
    assert frac < MAX_OFF_CHAIN


def test_one_live_row_in_the_last_tile_at_depth(M):
    """B*T = 128*256 + 1 at gpc = 7 through the C entry: the last tile's 127 clipped rows of each plane land neither
    before plane 0, after plane 4, nor (the contract over all five planes) in the next plane."""
    from rwkv_lm_ext_b200 import _lib
    lib = _lib.load()
    B, T, C = 3, 10923, 2048
    assert plan(B * T, C) == (257, 5, 7, 4)
    x, maa, h, w2, st = _inputs(B, T, C, True, seed=5)
    PAD = 128 * C                                          # a whole tile of rows on either side
    n = 5 * B * T * C
    buf = torch.full((n + 2 * PAD,), 7.0, dtype=torch.bfloat16, device=DEV)
    out = buf[PAD:PAD + n].view(5, B, T, C)
    p = _lib.ptr
    _lib.check(lib.tmix_ddlerp_lora_bf16(B, T, C, R, p(x), p(st), p(maa), p(h), p(w2), p(out),
                                         torch.cuda.current_stream().cuda_stream), "tmix_ddlerp_lora_bf16")
    torch.cuda.synchronize()
    assert bool((buf[:PAD] == 7.0).all()) and bool((buf[-PAD:] == 7.0).all())
    assert assert_ddlerp_contract(out, x, maa, h, w2, st, "tail") < MAX_OFF_CHAIN


def test_repeatable_and_the_same_on_any_stream(M):
    """The kernel has no atomics: at the 3B shape (14 groups per CTA) two launches are bit-identical, and so is a
    launch on a side stream.  A difference would be a race between an x refill or a W2 refill and the epilogue."""
    B, T, C = 16, 4096, 2560
    assert plan(B * T, C)[2] == 14
    x, maa, h, w2, st = _inputs(B, T, C, True, seed=7)
    a = M.tmix_ddlerp_lora(x, maa, h, w2, st)
    b = M.tmix_ddlerp_lora(x, maa, h, w2, st)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        c = M.tmix_ddlerp_lora(x, maa, h, w2, st)
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(a, b)
    assert torch.equal(a, c)


# ------------------------------------------------------------------------------------------------------------------
# ranks other than 32 (and C not a multiple of 64): bmm + tmix_ddlerp_mix
# ------------------------------------------------------------------------------------------------------------------
def _fp64_grads(leaves, go):
    """fp64 autograd on the GPU of x + xx * (maa_n + h_n @ W2_n) for the five output gradients go"""
    x, maa, h, w2, st = leaves
    B, T, C = x.shape
    rank = w2.shape[1]
    l64 = [t.detach().double().requires_grad_(True) if t is not None else None for t in leaves]
    prev = torch.zeros(B, 1, C, device=DEV, dtype=torch.float64) if st is None else l64[4].unsqueeze(1)
    xx = torch.cat([prev, l64[0][:, :-1]], 1) - l64[0]
    m = torch.bmm(l64[2].view(B * T, 5, rank).transpose(0, 1), l64[3]).view(5, B, T, C)
    ref = l64[0] + xx * (l64[1].view(5, 1, 1, C) + m)
    (ref * torch.stack(go).double()).sum().backward()
    return [l.grad if l is not None else None for l in l64]


def _relrms(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / (b.norm() + 1e-300)).item()


@pytest.mark.parametrize("rank,C", [(16, 768), (64, 4096), (32, 96)], ids=["R16", "R64", "C96"])
def test_other_shapes_take_the_bmm_route(M, rank, C):
    """Without grad: bit for bit bmm + tmix_ddlerp_mix.  With grad: the gradients of x, maa, h, W2 and the shift state
    against fp64 autograd, with the bounds of test_ddlerp_lora_fused."""
    B, T = 3, 130
    x, maa, h, w2, st = _inputs(B, T, C, True, seed=rank + C, rank=rank)
    got = M.tmix_ddlerp_lora(x, maa, h, w2, st)
    m = torch.bmm(h.view(B * T, 5, rank).transpose(0, 1), w2).view(5, B, T, C)
    assert torch.equal(got, M.tmix_ddlerp_mix(x, maa, m, st))
    leaves = [t.clone().requires_grad_(True) for t in (x, maa, h, w2, st)]
    outs = M.tmix_ddlerp_lora(*leaves[:4], leaves[4])
    g = torch.Generator(device=DEV).manual_seed(1)
    go = [torch.randn(B, T, C, generator=g, device=DEV).bfloat16() for _ in range(5)]
    torch.autograd.backward(list(outs), go)
    for name, a, want in zip(("gx", "gmaa", "gh", "gw2", "gshift"), leaves, _fp64_grads(leaves, go)):
        assert _relrms(a.grad, want) < 1.5e-2, name


# ------------------------------------------------------------------------------------------------------------------
# backward at the 1B6 training shape
# ------------------------------------------------------------------------------------------------------------------
DEPTH = (8, 4096, 2048)


@pytest.fixture(scope="module")
def depth_case():
    B, T, C = DEPTH
    x, maa, h, w2, st = _inputs(B, T, C, True, seed=11)
    g = torch.Generator(device=DEV).manual_seed(12)
    go = [torch.randn(B, T, C, generator=g, device=DEV).bfloat16() for _ in range(5)]
    return (x, maa, h, w2, st), go


def _grads(M, inputs, go, trainable=(True,) * 5, outputs=range(5), rows=None):
    """gradients of the five inputs from a backward through `outputs` only (the last of them cut to its first `rows`
    batch rows when given); None where an input is frozen"""
    leaves = [t.clone().requires_grad_(req) for t, req in zip(inputs, trainable)]
    outs = M.tmix_ddlerp_lora(*leaves[:4], leaves[4])
    ys = [outs[n] for n in outputs]
    gs = [go[n] for n in outputs]
    if rows is not None:
        ys[-1], gs[-1] = ys[-1][:rows], gs[-1][:rows]
    torch.autograd.backward(ys, gs)
    return [l.grad for l in leaves]


def test_backward_at_depth_against_fp64(M, depth_case):
    inputs, go = depth_case
    assert plan(DEPTH[0] * DEPTH[1], DEPTH[2])[2:] == (7, 4)
    got = _grads(M, inputs, go)
    for name, a, want in zip(("gx", "gmaa", "gh", "gw2", "gshift"), got, _fp64_grads(inputs, go)):
        assert a is not None and bool(torch.isfinite(a).all()), name
        rr = _relrms(a, want)
        err, top = (a.double() - want).abs().max().item(), want.abs().max().item()
        print(f"ddlerp_lora backward {name}: rel-RMS {rr:.3e}, max abs err {err:.3e} of max |ref| {top:.3e}")
        assert rr < 1e-2, f"{name}: rel-RMS {rr:.4g}"
        assert err <= 2.0 ** -7 * top, f"{name}: max abs err {err:.4g} vs max |ref| {top:.4g}"


def test_frozen_maa_and_w2_give_the_same_input_gradients(M, depth_case):
    """LoRA SFT and state tuning freeze time_maa_* and time_maa_w2: no gradient for them, and the gradients of x, h and
    the shift state bit-identical to the trainable run."""
    inputs, go = depth_case
    full = _grads(M, inputs, go)
    frozen = _grads(M, inputs, go, trainable=(True, False, True, False, True))
    assert frozen[1] is None and frozen[3] is None
    for name, i in (("gx", 0), ("gh", 2), ("gshift", 4)):
        assert torch.equal(frozen[i], full[i]), name


def test_outputs_without_a_gradient_count_as_zero(M, depth_case):
    """The bi-encoder feeds the gate only the plain half of the stacked batch (tmix_x060_project's gate_rows), and an
    output may be unused altogether: the gradients equal those of the same call given explicit zero gradients."""
    inputs, go = depth_case
    rows = DEPTH[0] // 2
    partial = _grads(M, inputs, go, outputs=(0, 2, 3, 4), rows=rows)        # no gradient for output 1, half of 4
    go0 = list(go)
    go0[1] = torch.zeros_like(go[1])
    go0[4] = go[4].clone()
    go0[4][rows:] = 0
    full = _grads(M, inputs, go0)
    for name, a, b in zip(("gx", "gmaa", "gh", "gw2", "gshift"), partial, full):
        assert torch.equal(a, b), name
