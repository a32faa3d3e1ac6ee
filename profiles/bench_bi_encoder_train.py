"""Training step of the bidirectional encoder (RwkvEncoder, semantics 2) at the 1B6 shape (synthetic.make_bi_encoder:
D2048, H32, FFN 7168, vocab 65536, full fine-tuning) over make_passages(64, T=512) (padded rows).

The loss is a workload, not a restatement of the reference's trainer: an in-batch contrastive loss over 32
(query, positive) pairs -- cosine similarity x 20, then cross-entropy.  Forward + backward, no optimizer.

Arms, alternated in one process:
  * fused: encoders.bi_encoder_encode (stack_reversed / groupnorm_gate_pair forward and backward kernels);
  * composition: the same model with bi_tmix_forward restated from the public pieces (torch.cat, reverse_x,
    groupnorm_gate), the route a training step took before the two backward kernels;
  each with checkpoint (block recomputation) on and off.
Reports ms per step and passages/s at `--layers` (default 8: the depth at which the no-checkpoint arms fit), the
checkpointed fused step at 24 layers, peak torch.cuda.max_memory_allocated above the weights for L = 2 and L = 8 (growth
per layer), and the two new kernels' time and achieved bytes/s at 64 x 512 x 2048 against MEASURED_PEAKS.json (when it
is there) and a device-to-device copy measured in the same run.  The card's name and power limit are read in the same
run.  Prints one JSON line; `--out FILE` also writes it there.
usage: python profiles/bench_bi_encoder_train.py [--layers L] [--steps K] [--out FILE]"""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.nn.functional as F
import rwkv_lm_ext_b200 as M
from rwkv_lm_ext_b200 import _lib, encoders, heads, ops, tmix
from rwkv_lm_ext_b200.synthetic import make_bi_encoder, make_passages

B, T, D, H = 64, 512, 2048, 32


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def composition_bi_tmix(att, x, rev_idx):
    """bi_tmix_forward composed from the differentiable public pieces (the route before the fused backward kernels)."""
    B_, T_, C = x.shape
    Hh = att.time_faaaa.shape[0]
    xx = torch.cat([x, heads.reverse_x(x, rev_idx)], 0)
    r, k, v, g, w = tmix.tmix_x060_project(att, xx, gate_rows=B_)
    y2 = ops.RUN_CUDA_RWKV6(2 * B_, T_, C, Hh, r, k, v, w, att.time_faaaa)
    y, ry = y2[:B_], y2[B_:]
    z = heads.groupnorm_gate((y + heads.reverse_x(ry, rev_idx)) / 2, g, att.ln_x.weight, att.ln_x.bias, Hh, att.ln_x.eps,
                             gate_act="silu")
    return att.output(z)


def encode(model, idx, fused, checkpoint):
    if fused:
        return encoders.bi_encoder_encode(model, idx, checkpoint=checkpoint)
    _, rev = heads.create_mask_and_rev_idx(idx, 1, 0)
    hidden = encoders.blocks_forward(model.blocks, model.emb(idx), model.ln_out,
                                     lambda blk, h: composition_bi_tmix(blk.att, h, rev), checkpoint)
    return heads.eos_gather(hidden.contiguous(), idx, 1)[0]


def contrastive_loss(emb, scale=20.0):
    n = emb.shape[0] // 2
    e = F.normalize(emb.float(), dim=-1)
    return F.cross_entropy(e[:n] @ e[n:].T * scale, torch.arange(n, device=emb.device))


def step(model, idx, fused, checkpoint):
    model.zero_grad(set_to_none=True)
    loss = contrastive_loss(encode(model, idx, fused, checkpoint))
    loss.backward()
    return loss


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


ARMS = [(True, False), (False, False), (True, True), (False, True)]
NAME = {(True, False): "fused", (False, False): "composition", (True, True): "fused_checkpoint",
        (False, True): "composition_checkpoint"}


def steps_and_memory(layers, steps, idx, arms=ARMS, memory=True):
    model = make_bi_encoder(layers=layers, seed=0, device="cuda")
    model.train()
    for arm in arms:                                                   # warm-up (and every .grad allocated once)
        step(model, idx, *arm)
    out = {a: {"ms": [], "loss": None, "peak_bytes": None} for a in arms}
    for _ in range(steps):                                             # alternate the arms
        for arm in arms:
            out[arm]["ms"].append(timed(lambda: step(model, idx, *arm), 1))
    for arm in arms:
        model.zero_grad(set_to_none=True)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()                           # weights (gradients are set to None)
        torch.cuda.reset_peak_memory_stats()
        out[arm]["loss"] = float(step(model, idx, *arm))
        torch.cuda.synchronize()
        out[arm]["peak_bytes"] = torch.cuda.max_memory_allocated() - base
    params = sum(p.numel() for p in model.parameters())
    del model
    torch.cuda.empty_cache()
    return out, params


def kernel_times(peak_gbs):
    """The two new kernels at 64 x 512 x 2048 (every operand larger than the 126 MB L2)."""
    lib = _lib.load()
    g_ = torch.Generator(device="cuda").manual_seed(0)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=g_).bfloat16()
    idx = make_passages(B, T=T, seed=0).cuda()
    _, rev = heads.create_mask_and_rev_idx(idx, 1, 0)
    y2, g, gout, lw, lb = rnd(2 * B, T, D), rnd(B, T, D), rnd(B, T, D), rnd(D), rnd(D)
    gy2, gg = torch.empty_like(y2), torch.empty_like(g)
    gw, gb = torch.empty(D, device="cuda"), torch.empty(D, device="cuda")
    ws = heads._ws(lib, B, T, D, 2, y2.device)
    s = torch.cuda.current_stream().cuda_stream
    p = lambda t: t.data_ptr()

    def pair():
        lib.groupnorm_gate_pair_backward_bf16(B, T, D, H, 1e-5 * 64, 1, p(y2), p(y2[B:]), p(rev), p(g), p(lw), p(lb), p(gout),
                                              p(gy2), p(gy2[B:]), p(gg), p(gw), p(gb), p(ws), ws.numel(), s)

    gxx, gx = rnd(2 * B, T, D), torch.empty(B, T, D, device="cuda", dtype=torch.bfloat16)

    def stack():
        lib.stack_reversed_backward_bf16(B, T, D, p(gxx), p(rev), p(gx), s)

    copy_src = rnd(4 * B, T, D)
    copy_dst = torch.empty_like(copy_src)
    n = B * T * D
    res = {}
    for name, fn, nbytes in (("groupnorm_gate_pair_backward_bf16", pair, 14 * n + 8 * B * T),
                             ("stack_reversed_backward_bf16", stack, 6 * n + 8 * B * T),
                             ("device_copy_reference", lambda: copy_dst.copy_(copy_src), 2 * copy_src.numel() * 2)):
        for _ in range(5):
            fn()
        ms = min(timed(fn, 50) for _ in range(3))
        res[name] = {"us": round(ms * 1e3, 1), "bytes": nbytes, "GB_per_s": round(nbytes / (ms * 1e-3) / 1e9, 1)}
        if peak_gbs:
            res[name]["of_measured_peak"] = round(res[name]["GB_per_s"] / peak_gbs, 3)
    # the same two pieces through autograd, fused against the composition (op level, forward + backward)
    yl = y2.clone().requires_grad_(True)
    gl = g.clone().requires_grad_(True)
    wl, bl = lw.clone().requires_grad_(True), lb.clone().requires_grad_(True)

    def pair_op(fused):
        if fused:
            out = heads.groupnorm_gate_pair(yl, None, rev, gl, wl, bl, H, 1e-5 * 64, "silu")
        else:
            out = heads.groupnorm_gate((yl[:B] + heads.reverse_x(yl[B:], rev)) / 2, gl, wl, bl, H, 1e-5 * 64, "silu")
        out.backward(gout)

    xl = rnd(B, T, D).requires_grad_(True)

    def stack_op(fused):
        out = heads.stack_reversed(xl, rev) if fused else torch.cat([xl, heads.reverse_x(xl, rev)], 0)
        out.backward(gxx)

    for name, fn in (("groupnorm_gate_pair_fwd_bwd", pair_op), ("stack_reversed_fwd_bwd", stack_op)):
        ms = {True: [], False: []}
        for f in (True, False):
            fn(f)
        for _ in range(3):
            for f in (True, False):
                ms[f].append(timed(lambda: fn(f), 20))
        res[name] = {"fused_us": round(min(ms[True]) * 1e3, 1), "composition_us": round(min(ms[False]) * 1e3, 1)}
    return res


def main(layers=8, steps=3):
    M.load()
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak_gbs = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else None
    idx = make_passages(B, T=T, seed=0).cuda()
    res = {"card": card(), "config": f"1B6 bi-encoder (D{D} H{H} FFN7168 vocab65536), full fine-tuning, "
                                     f"{B} passages x {T} tokens (padded rows), contrastive loss over {B // 2} pairs, "
                                     "forward + backward, no optimizer", "measured_peak_hbm_gbs": peak_gbs}
    res["kernels_64x512x2048"] = kernel_times(peak_gbs)
    arms, params = steps_and_memory(layers, steps, idx)
    res[f"L{layers}"] = {NAME[a]: {"ms_per_step": [round(x, 1) for x in v["ms"]],
                                   "passages_per_s": round(B / (min(v["ms"]) * 1e-3), 1),
                                   "peak_bytes_above_weights": v["peak_bytes"], "loss": v["loss"]} for a, v in arms.items()}
    res[f"L{layers}"]["params"] = params
    small, _ = steps_and_memory(2, 1, idx)
    res["peak_growth_per_layer_L2_to_L%d_bytes" % layers] = {
        NAME[a]: round((arms[a]["peak_bytes"] - small[a]["peak_bytes"]) / (layers - 2)) for a in ARMS}
    res["L2_peak_bytes_above_weights"] = {NAME[a]: small[a]["peak_bytes"] for a in ARMS}
    res["boundary_tensor_bytes"] = B * T * D * 2
    res["wkv_chunk_state_bytes_per_layer"] = int(_lib.load().wkv6_saved_bytes(2 * B, T, D, H))
    full, params24 = steps_and_memory(24, steps, idx, arms=[(True, True), (False, True)])
    res["L24"] = {NAME[a]: {"ms_per_step": [round(x, 1) for x in v["ms"]], "passages_per_s": round(B / (min(v["ms"]) * 1e-3), 1),
                            "peak_bytes_above_weights": v["peak_bytes"], "loss": v["loss"]} for a, v in full.items()}
    res["L24"]["params"] = params24
    res["card_after"] = card()
    return res


if __name__ == "__main__":
    L = int(sys.argv[sys.argv.index("--layers") + 1]) if "--layers" in sys.argv else 8
    K = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 3
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    line = json.dumps(main(layers=L, steps=K))
    print(line)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(line + "\n")
