"""BASELINE config 5 at the model level: one training step of a 3B-shape RWKV-6 (L32, D2560, H40, FFN 8960,
vocab 65536, full fine-tuning, `init_like_reference` weights) over B = 1 sequence of 16 x 4096 synthetic tokens,
chunk by chunk with the fp32 WKV-state carry (infctx.infctx_train_step).  Reports, for the truncated gradient
(exact=False, the reference's semantics) and the exact one (exact=True):
  * tokens/s of forward + backward (CUDA events around whole steps, alternating the two modes);
  * peak torch.cuda.max_memory_allocated above the model and its gradients, at 4 and at 16 chunks of 4096 tokens,
    next to the bytes of the chunk-start states the driver keeps (the only part that grows with the chunk count);
  * the driver's first sweep (the layers over the first 15 chunks, states only) as it runs, with autograd enabled so
    that it takes the training pair's segment plan, against the same sweep under no_grad.
The card's name, power limit and max SM clock are read in the same run.  Prints one JSON line; `--out FILE` also
writes it there.  usage: python profiles/bench_infctx_model.py [--layers L] [--steps K] [--out FILE]"""
import json, os, subprocess, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import rwkv_lm_ext_b200 as M
from rwkv_lm_ext_b200 import sft


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def main(layers=32, D=2560, H=40, ffn=8960, vocab=65536, chunk=4096, n_chunks=16, steps=2):
    dev = torch.device("cuda", 0)
    M.load()
    t_init = time.time()
    with torch.device("meta"):
        model = sft.RwkvSft(layers, D, H, ffn, vocab, train_type="full")
    model = model.to_empty(device=dev).bfloat16()
    sft.init_like_reference(model, seed=0)
    t_init = time.time() - t_init
    n_params = sum(p.numel() for p in model.parameters())
    g = torch.Generator().manual_seed(0)
    ids = torch.randint(0, vocab, (1, n_chunks * chunk + 1), generator=g).to(dev)
    idx, tgt = ids[:, :-1].contiguous(), ids[:, 1:].contiguous()

    def step(exact, n=n_chunks):
        loss, _ = M.infctx_train_step(model, idx[:, :n * chunk], tgt[:, :n * chunk], chunk, exact=exact)
        return loss

    res = {"card": card(), "config": f"RWKV-6 3B shape L{layers} D{D} H{H} FFN{ffn} vocab{vocab}, full fine-tuning, "
                                     f"B=1, {n_chunks} x {chunk} tokens, fp32 WKV-state carry",
           "params": n_params, "init_s": round(t_init, 1)}
    for exact in (False, True):                            # warm-up of both modes (and every parameter's .grad)
        step(exact)
    ms = {False: [], True: []}
    losses = {}
    for rep in range(steps):                               # alternate the two modes
        for exact in (False, True):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            loss = step(exact)
            b.record()
            torch.cuda.synchronize()
            ms[exact].append(a.elapsed_time(b))
            losses[exact] = float(loss)
    tokens = n_chunks * chunk
    for exact in (False, True):
        key = "exact" if exact else "truncated"
        res[key] = {"ms_per_step": [round(x, 1) for x in ms[exact]], "tokens_per_s": round(tokens / (min(ms[exact]) * 1e-3)),
                    "loss": losses[exact]}
    res["exact_over_truncated"] = round(min(ms[True]) / min(ms[False]), 3)
    # first sweep: autograd enabled (what the driver runs) against no_grad
    from rwkv_lm_ext_b200.infctx import _chunk_hidden

    def sweep1(grad):
        st = M.BlockStateList.create(layers, 1, D, H, dev, torch.bfloat16, wkv_dtype=torch.float32)
        w, a, f = (list(t.unbind(0)) for t in (st.wkv_states, st.shift_states[:, 0], st.shift_states[:, 1]))
        with torch.enable_grad() if grad else torch.no_grad():
            for c in range(n_chunks - 1):
                lv = [[x.detach().requires_grad_(grad) for x in lst] for lst in (w, a, f)]
                h, w, a, f = _chunk_hidden(model, idx[:, c * chunk:(c + 1) * chunk], *lv, False)
                w, a, f = ([x.detach() for x in lst] for lst in (w, a, f))
                del h, lv

    s1 = {True: [], False: []}
    for rep in range(steps):
        for grad in (True, False):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            sweep1(grad)
            b.record()
            torch.cuda.synchronize()
            s1[grad].append(a.elapsed_time(b))
    res["sweep1_ms_autograd"] = round(min(s1[True]), 1)
    res["sweep1_ms_no_grad"] = round(min(s1[False]), 1)
    # peak memory above the weights and their gradients (allocated before the baseline is read)
    boundary = layers * H * 64 * 64 * 4 + layers * 2 * D * 2
    res["boundary_state_bytes"] = boundary
    for exact in (False, True):
        key = "exact" if exact else "truncated"
        for n in (4, n_chunks):
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            step(exact, n)
            torch.cuda.synchronize()
            res[key][f"peak_bytes_above_weights_{n}_chunks"] = torch.cuda.max_memory_allocated() - base
        res[key]["peak_growth_4_to_16_chunks_bytes"] = (res[key][f"peak_bytes_above_weights_{n_chunks}_chunks"]
                                                       - res[key]["peak_bytes_above_weights_4_chunks"])
    res["stored_boundaries_growth_4_to_16_chunks_bytes"] = (n_chunks - 4) * boundary
    res["weights_and_grads_bytes"] = 2 * 2 * n_params
    return res


if __name__ == "__main__":
    L = int(sys.argv[sys.argv.index("--layers") + 1]) if "--layers" in sys.argv else 32
    K = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 2
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    line = json.dumps(main(layers=L, steps=K))
    print(line)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(line + "\n")
