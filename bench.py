#!/usr/bin/env python
"""bench.py -- WKV6 fwd+bwd tokens/s at the RWKV-6 1B6 shape (BASELINE.json configs[1]), and -- in the
same JSON line, key "bi_encoder" -- BASELINE metric (ii): bi-encoder passages/s at the 1B6 shape (configs[2]),
batch-sharded over the ranks with one NCCL all_gather of the [B_local, D] embeddings per step.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one forward + backward pass of the WKV6 operator over one batch of synthetic input
(B=8, T=4096, H=32, N=64, bf16) per GPU, through the reference-shaped Python surface
(RUN_CUDA_RWKV6 -> C ABI -> sm_100a kernels).  N > 1 is launched by torchrun, one rank per GPU;
the batch dimension is sharded, there is no data-path collective (weak scaling).

Prints ONE JSON line (rank 0).  `value` = device-resident throughput; `e2e` = same metric with host
buffers (pinned) copied in and results copied out inside the timed region; `roofline` = achieved
algorithmic HBM bytes/s of the dominant kernel over the measured copy bandwidth
(MEASURED_PEAKS.json); `cpu_baseline` = the oracle's C port (oracle/wkv6_oracle.c, the reference
kernels' arithmetic on host cores) on a bounded sample; `reference_cuda` = the reference's own CUDA
kernels (oracle/_ref) timed on the same GPU and inputs, when they were built.
`--impl reference` times the reference's CPU implementation of the path (the oracle port, all host
threads) on a bounded sample of the same workload.
`--dump-outputs DIR` writes what the last timed step returned (rank 0) as DIR/<name>.npy, float32: a fixed sample of
y, gr, gk, gv, gw (the same elements in every run, see dump_index) and the whole gu.  The inputs depend on nothing but
the arguments, so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "WKV6 fwd+bwd tokens/s (1B6 shape)"
UNIT = "tokens/s"
B, T, H, N = 8, 4096, 32, 64
C = H * N
BYTES_FWD = 10     # r,k,v,w read + y written, bf16                      (SURVEY.md 8d)
BYTES_BWD = 18     # r,k,v,w,gy read + gr,gk,gv,gw written, bf16
CPU_SAMPLE = dict(B=1, T=4096, H=32)   # 1/8 of one step's batch
DUMP_SAMPLE = 1 << 21                  # elements dumped of each [B, T, C] output: 8 MB of float32 each, 40 MB in all


def dump_index(device="cpu"):
    """Sorted, distinct flat indices into a [B, T, C] output: one element of every run of B*T*C / DUMP_SAMPLE
    consecutive ones, its offset in the run drawn by a generator with a fixed seed."""
    import torch
    run = B * T * C // DUMP_SAMPLE
    assert run * DUMP_SAMPLE == B * T * C
    g = torch.Generator().manual_seed(0)
    return (torch.arange(DUMP_SAMPLE) * run + torch.randint(0, run, (DUMP_SAMPLE,), generator=g)).to(device)


def dump_outputs(out_dir, y, grads):
    """Writes one step's results of RUN_CUDA_RWKV6 + backward: y and gr, gk, gv, gw sampled at dump_index(), gu whole."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    idx = dump_index(y.device)
    for name, t in zip(("y", "gr", "gk", "gv", "gw"), [y] + list(grads[:4])):
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().reshape(-1)[idx].float().cpu().numpy())
    np.save(os.path.join(out_dir, "gu.npy"), grads[4].detach().float().cpu().numpy())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def config(n_gpus):
    return {"workload": f"WKV6 op fwd+bwd, B={B} T={T} H={H} N={N} per GPU (RWKV-x060 World 1B6 shape), "
                        "w ~ time_decay range U(-6,-1)+0.3N(0,1), synthetic randn r/k/v/gy",
            "global_batch": B * n_gpus, "seq_len": T, "heads": H, "head_size": N,
            "parallelism": f"batch-sharded x{n_gpus}, no data-path collective",
            "l2": "inputs (6 x 134 MB per step) are larger than the 126 MB L2; no explicit flush"}


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self._nv = self._h = None
        try:            # NVML is initialised here, before the timed region, so that sampling starts with it
            import pynvml as nv
            nv.nvmlInit()
            self._nv, self._h = nv, nv.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
        except Exception as e:  # no NVML: report that instead of inventing numbers
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def run(self):
        nv, h = self._nv, self._h
        if nv is None:
            return
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "sw_thermal_slowdown": 0x20,
                 "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80, "sync_boost": 0x10,
                 "applications_clocks": 0x2}
        try:
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    bits = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    bits = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, b in names.items():
                    if bits & b:
                        self.reasons.add(k)
                time.sleep(0.005)
        except Exception as e:
            self.reasons.add(f"nvml_error:{type(e).__name__}")

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def run_cpu(steps, warmup, budget_s=20.0, exact_steps=False):
    """The oracle's C port on host cores, on CPU_SAMPLE.  Default (the `cpu_baseline` leg of our own arm): up to `steps`
    runs of the sample, stopping early once `budget_s` seconds of CPU work are spent.  exact_steps (the reference arm):
    `warmup` untimed and EXACTLY `steps` timed runs; if they would not fit in `budget_s`, the sample's T is halved until
    they do.  Returns (tokens/s, cores, s/run, runs, T of the sample)."""
    from oracle import c_oracle
    from rwkv_lm_ext_b200.synthetic import make_inputs
    s = CPU_SAMPLE
    r, k, v, w, u, gy = (t.float() for t in make_inputs(s["B"], s["T"], s["H"], seed=0, decay="model"))
    cores = c_oracle.use_all_cores()
    Ts = s["T"]

    def one(n):
        c_oracle.forward(r[:, :n], k[:, :n], v[:, :n], w[:, :n], u)
        c_oracle.backward(r[:, :n], k[:, :n], v[:, :n], w[:, :n], u, gy[:, :n])

    if exact_steps:
        one(256)
        t0 = time.perf_counter()
        one(Ts)
        est = time.perf_counter() - t0
        while Ts > 256 and est * (steps + warmup) > budget_s:
            Ts //= 2
            est /= 2
        r, k, v, w, gy = (t[:, :Ts].contiguous() for t in (r, k, v, w, gy))
        for _ in range(warmup):
            one(Ts)
    else:
        for _ in range(warmup):
            one(256)
    ts = []
    while len(ts) < steps and (exact_steps or not ts or sum(ts) < budget_s):
        t0 = time.perf_counter()
        one(Ts)
        ts.append(time.perf_counter() - t0)
    sec = sum(ts) / len(ts)
    return s["B"] * Ts / sec, cores, sec, len(ts), Ts


def run_reference_python(budget_s=12.0):
    """The reference's OWN CPU implementation of the recurrence, unmodified: run_rwkv6_forward of
    src/model_encoder_run.py:31-62 (= tests/test_cpu.py:42-73), from baseline/_ref (placed there by
    __graft_entry__.build(); git-ignored).  It is forward only (in-place state updates: no autograd) and a Python
    loop over T x 64, so it is timed on the WKV6 call of BASELINE configs[0] (169M shape: B=8, T=512, H=12, fp32),
    bounded by `budget_s`.  Returns None when the file is not there."""
    import importlib.util
    path = os.path.join(ROOT, "baseline", "_ref", "src", "model_encoder_run.py")
    if not os.path.isfile(path):
        return None
    os.environ.setdefault("RWKV_HEAD_SIZE_A", "64")
    os.environ["NO_CUDA"] = "1"
    import torch
    from rwkv_lm_ext_b200.synthetic import make_inputs
    spec = importlib.util.spec_from_file_location("_ref_model_encoder_run", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    Br, Tr, Hr = 8, 512, 12
    r, k, v, w, u, _ = (t.float() for t in make_inputs(Br, Tr, Hr, seed=0, decay="model"))
    torch.set_num_threads(os.cpu_count() or 1)
    n = 32                                         # time a prefix first: the loop is linear in T
    t0 = time.perf_counter()
    with torch.no_grad():
        mod.run_rwkv6_forward(r[:, :n].contiguous(), k[:, :n].contiguous(), v[:, :n].contiguous(), w[:, :n].contiguous(), u)
    per_tok = (time.perf_counter() - t0) / n
    Tt = int(max(n, min(Tr, budget_s / per_tok)))
    t0 = time.perf_counter()
    with torch.no_grad():
        y = mod.run_rwkv6_forward(r[:, :Tt].contiguous(), k[:, :Tt].contiguous(), v[:, :Tt].contiguous(), w[:, :Tt].contiguous(), u)
    sec = time.perf_counter() - t0
    return {"what": "reference run_rwkv6_forward (src/model_encoder_run.py:31-62, unmodified, from baseline/_ref), "
                    f"forward only, fp32, B={Br} T={Tt} H={Hr} (configs[0] shape{'' if Tt == Tr else ', first ' + str(Tt) + ' tokens'})",
            "seconds": sec, "tokens_per_s_forward": Br * Tt / sec, "cores": os.cpu_count(), "kind": "reference",
            "_y": y, "_inputs": (r[:, :Tt].contiguous(), k[:, :Tt].contiguous(), v[:, :Tt].contiguous(), w[:, :Tt].contiguous(), u)}


BI = dict(layers=24, D=2048, H=32, ffn=7168, vocab=65536, micro_batch=64, T=512)   # SURVEY.md 8(d) config 3


def run_bi_encoder(args, M, torch, dist, dev, rank, world, barrier):
    """BASELINE metric (ii): corpus embedding with the bidirectional 1B6 encoder (src/model_encoder_run.py:296-350,
    semantics 2 of SURVEY.md 2.3), 512-token padded passages, micro-batch 64 per GPU, forward only.
    value  : passages/s, ids resident on the device, all_gather of the embeddings inside the timed region
    e2e    : the call a user makes: token ids in pinned host memory -> embeddings of ALL ranks in pinned host memory
    accuracy (1 GPU only): the same 1024 passages on the exact SIMT route; min cosine and top-1 neighbour agreement"""
    from rwkv_lm_ext_b200.synthetic import make_bi_encoder, make_passages
    c = BI
    model = make_bi_encoder(c["layers"], c["D"], c["H"], c["ffn"], c["vocab"], seed=0, device=dev)
    Bm, T, D = c["micro_batch"], c["T"], c["D"]
    ids_host = make_passages(Bm, T, c["vocab"], seed=100 + rank).pin_memory()
    ids = ids_host.to(dev)
    gathered = torch.empty(world * Bm, D, dtype=torch.bfloat16, device=dev)
    out_host = torch.empty(world * Bm, D, dtype=torch.bfloat16).pin_memory()

    # the forward of one micro-batch shape as a CUDA-graph replay (rwkv_lm_ext_b200.GraphedForward): ~3 k launches per
    # step, launched eagerly the GPU waits for the host between the short ones
    # (opt-in: measured 121.9 ms against 122.9 ms eager -- at 64 x 512 tokens per step the host keeps ahead of the GPU)
    enc = M.GraphedForward(M.bi_encoder_encode, model, ids) if args.bi_graph else None

    def step(idx, eager=False):
        if enc is None or eager:
            with torch.no_grad():
                e = M.bi_encoder_encode(model, idx)                 # [Bm, D] bf16
        else:
            e = enc(idx)                                            # idx: device or pinned host ids (copied into the graph's input)
        if world > 1:
            dist.all_gather_into_tensor(gathered, e.contiguous())   # the one data-path collective of this config
            return gathered
        return e

    def step_e2e():
        e = step(ids_host if enc is not None else ids_host.to(dev, non_blocking=True))
        out_host[: e.size(0)].copy_(e, non_blocking=True)

    def timed(fn, n):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        barrier()
        ms = a.elapsed_time(b) / n
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    steps = max(3, min(args.steps, 10))
    for _ in range(3):
        step(ids)
    n0 = M.launch_count()
    ms = timed(lambda: step(ids), steps)
    launches = M.launch_count() - n0
    for _ in range(2):
        step_e2e()
    ems = timed(step_e2e, steps)
    eager_ms = ms
    if enc is not None:
        n0 = M.launch_count()
        eager_ms = timed(lambda: step(ids, eager=True), steps)
        launches = M.launch_count() - n0          # a replay launches the same kernels; the host-side counter only sees eager calls
    # Linears per layer: r, k, v for both directions, gate and output once (time mix); key, value, receptance (channel mix)
    lin_flops = 2 * Bm * T * c["layers"] * (8 * D * D + 2 * D * c["ffn"] + D * D)
    res = {"metric": "bi-encoder passages/s (1B6 shape)", "value": world * Bm / (ms * 1e-3), "unit": "passages/s",
           "ms_per_step": ms, "steps": steps, "micro_batch_per_gpu": [Bm, T], "global_batch": world * Bm,
           "model": f"RWKV-6 1B6 shape L{c['layers']} D{D} H{c['H']} FFN{c['ffn']}, random init, bf16",
           "scaling": "weak", "collective": "none" if world == 1 else f"all_gather [{Bm},{D}] bf16 per rank per step (NCCL)",
           "all_gather_bytes_per_step": 0 if world == 1 else world * Bm * D * 2,
           "linear_tflops_per_gpu": lin_flops / (ms * 1e-3) / 1e12, "gpu_launches": int(launches),
           "launch": "eager" if enc is None else "CUDA-graph replay of the whole forward (GraphedForward)",
           "eager": {"value": world * Bm / (eager_ms * 1e-3), "ms_per_step": eager_ms},
           "e2e": {"value": world * Bm / (ems * 1e-3), "unit": "passages/s", "ms_per_step": ems,
                   "h2d_bytes_per_step": Bm * T * 8, "d2h_bytes_per_step": world * Bm * D * 2,
                   "api": "rwkv_lm_ext_b200.bi_encoder_encode(model, idx): token ids in pinned host memory -> "
                          "embeddings of the whole global batch in pinned host memory"}}
    if world == 1:
        # accuracy gate of SURVEY 8(d) config 3 on 1024 passages: fused tensor-core route vs the exact SIMT WKV6 route
        n_mb = 16
        batches = [make_passages(Bm, T, c["vocab"], seed=500 + i).to(dev) for i in range(n_mb)]
        with torch.no_grad():
            ef = torch.cat([M.bi_encoder_encode(model, b) for b in batches]).float()
            M.set_impl("simt")
            try:
                es = torch.cat([M.bi_encoder_encode(model, b) for b in batches]).float()
            finally:
                M.set_impl(args.kernel_impl)
        cos = torch.nn.functional.cosine_similarity(ef, es, dim=-1)

        def top1(e):
            e = torch.nn.functional.normalize(e - e.mean(0, keepdim=True), dim=-1)     # centred: random-init embeddings share a large common component
            sim = e @ e.t()
            sim.fill_diagonal_(-2.0)
            return sim.argmax(-1)
        res["accuracy"] = {"passages": n_mb * Bm, "min_cosine_vs_exact_route": float(cos.min().item()),
                           "top1_neighbour_agreement": float((top1(ef) == top1(es)).float().mean().item()),
                           "what": "fused kernels + tcgen05 WKV6 vs the same forward with the exact fp32 SIMT WKV6 kernels"}
    del model
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--kernel-impl", default="auto", choices=["auto", "simt", "tc"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eager-step", action="store_true", help="time Python-launched steps instead of CUDA-graph replays of the step")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-bi-encoder", action="store_true")
    ap.add_argument("--bi-graph", action="store_true", help="bi-encoder leg as a CUDA-graph replay of the whole forward")
    ap.add_argument("--no-sft", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank != 0:
            return 0
        # same K and W as our arm; a step = one bounded sample of the workload (one batch row of the 8, shortened if K of
        # them would not fit in two minutes), timed as it is -- ms_per_step is the sample's own time, not an extrapolation
        warm = max(args.warmup, 3)
        val, cores, sec, steps, Ts = run_cpu(max(1, args.steps), warm, budget_s=120.0, exact_steps=True)
        sample = (f"fwd+bwd on B={CPU_SAMPLE['B']} T={Ts} H={CPU_SAMPLE['H']} per step "
                  f"({CPU_SAMPLE['B'] * Ts} of the workload's {B * T} tokens), mean of {steps} steps, {sec:.3f} s each, {cores} threads")
        line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
                "steps": steps, "warmup": warm, "ms_per_step": sec * 1e3, "tokens_per_step": CPU_SAMPLE["B"] * Ts,
                "full_step_ms_extrapolated": sec * 1e3 * (B * T) / (CPU_SAMPLE["B"] * Ts),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config(args.gpus),
                "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
                "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        rp = run_reference_python(budget_s=20.0)          # the reference's own (forward-only) CPU code, beside the port
        if rp:
            line["reference_python"] = {k_: v_ for k_, v_ in rp.items() if not k_.startswith("_")}
        print(json.dumps(line), flush=True)
        return 0

    import torch
    import torch.distributed as dist
    import rwkv_lm_ext_b200 as M
    from rwkv_lm_ext_b200.synthetic import make_inputs

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    M.load()
    M.set_impl(args.kernel_impl)

    # synthetic inputs, created on the host (pinned) so the e2e leg has real host buffers
    host = [t.pin_memory() for t in make_inputs(B, T, H, seed=rank, decay="model")]
    r, k, v, w, u, gy = (t.to(dev, non_blocking=True) for t in host)
    torch.cuda.synchronize()

    def step(r, k, v, w, u, gy, ev=None):
        leaves = [t.detach().requires_grad_(True) for t in (r, k, v, w, u)]
        if ev:
            ev[0].record()
        y = M.RUN_CUDA_RWKV6(B, T, C, H, *leaves)
        if ev:
            ev[1].record()
        y.backward(gy)
        if ev:
            ev[2].record()
        grads = [t.grad for t in leaves]
        for t in leaves:
            t.grad = None
        return y, grads

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step(r, k, v, w, u, gy)
    # The step (memset + forward kernel + backward kernel) is launch-bound for the host at 0.6 ms: with 8 ranks sharing
    # the box's cores the eager Python path costs up to 8 % of the step.  The operator has no host synchronisation and
    # takes its scratch from torch's allocator, so the step is captured ONCE into a CUDA graph and the timed region
    # replays it K times (same kernels, same buffers; tests/test_gpu_parity.py::test_cuda_graph_capture_fwd_bwd holds
    # replays bit-identical to eager calls).  --eager-step keeps the Python launches in the timed region instead.
    graph, launches_per_step = None, None
    if not args.eager_step:
        try:
            static = [t.detach().requires_grad_(True) for t in (r, k, v, w, u)]
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    M.RUN_CUDA_RWKV6(B, T, C, H, *static).backward(gy)
            torch.cuda.current_stream().wait_stream(side)
            for t in static:
                t.grad = None
            graph = torch.cuda.CUDAGraph()
            n0 = M.launch_count()
            with torch.cuda.graph(graph):
                y_static = M.RUN_CUDA_RWKV6(B, T, C, H, *static)
                y_static.backward(gy)
            launches_per_step = M.launch_count() - n0
            for _ in range(max(args.warmup, 10)):     # W untimed warm-up steps of the thing that is timed
                graph.replay()
        except Exception as e:                       # capture refused: time the eager step
            sys.stderr.write(f"bench: CUDA-graph capture of the step failed ({type(e).__name__}: {e}); timing eager steps\n")
            graph = None
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = M.launch_count()
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    if graph is not None:
        for i in range(args.steps):
            graph.replay()
        last = (y_static, [t.grad for t in static])
    else:
        for i in range(args.steps):
            last = step(r, k, v, w, u, gy)
    t_end.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    del last
    launches = launches_per_step * args.steps if graph is not None else M.launch_count() - launches0
    ms = t_start.elapsed_time(t_end) / args.steps
    eager_ms = ms
    if graph is not None:                            # the same K steps launched from Python, for the record
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            step(r, k, v, w, u, gy)
        e1.record()
        barrier()
        eager_ms = e0.elapsed_time(e1) / args.steps
    # forward / backward split (the roofline's per-launch duration): the same steps again with an event between the two
    # calls -- kept out of the timed region above, which holds exactly K steps and nothing else
    n_split = max(3, min(args.steps, 20))
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(n_split)]
    for i in range(n_split):
        step(r, k, v, w, u, gy, evs[i])
    barrier()
    fwd_ms = statistics.mean(e[0].elapsed_time(e[1]) for e in evs)
    bwd_ms = statistics.mean(e[1].elapsed_time(e[2]) for e in evs)
    if world > 1:
        tms = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    value = world * B * T / (ms * 1e-3)

    # ---- SURVEY 8(d)'s second run of this config: the reference tests' own decay distribution, w ~ N(0,1)
    # (tests/test_cpu.py:266), same shapes, same call; how many (b,h) streams left the tensor-core kernels
    w_randn = make_inputs(B, T, H, seed=1000 + rank, decay="randn")[3].to(dev)
    with M.exact_route_report() as rep:
        for _ in range(3):
            step(r, k, v, w_randn, u, gy)
    rn_steps = max(3, min(args.steps, 20))
    barrier()
    a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a_.record()
    for _ in range(rn_steps):
        step(r, k, v, w_randn, u, gy)
    b_.record()
    barrier()
    rn_ms = a_.elapsed_time(b_) / rn_steps
    if world > 1:
        tms = torch.tensor([rn_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        rn_ms = float(tms.item())
    randn_decay = {"ms_per_step": rn_ms, "value": world * B * T / (rn_ms * 1e-3), "unit": UNIT, "steps": rn_steps,
                   "exact_route_streams": rep.streams()[0], "streams": rep.streams()[1] // 3,
                   "slowdown_vs_model_decay": rn_ms / ms, "what": "same op and shape with w ~ N(0,1)"}
    del w_randn

    # ---- end to end: host buffers in, results out, inside the timed region.  Three CUDA streams form
    # the pipeline a data-parallel worker would run: copy-in of step i+1 and copy-out of step i-1
    # overlap the kernels of step i (PCIe is full duplex); every step still moves all of its inputs
    # from pinned host memory and all of its results back.
    e2e = None
    if not args.no_e2e:
        NBUF = 2
        outs_host = [[torch.empty(B, T, C, dtype=torch.bfloat16).pin_memory() for _ in range(5)] for _ in range(NBUF)]
        gu_host = [torch.empty(H, N, dtype=torch.bfloat16).pin_memory() for _ in range(NBUF)]
        dev_in = [[torch.empty_like(t, device=dev) for t in host] for _ in range(NBUF)]
        h2d = sum(t.numel() * t.element_size() for t in host)
        d2h = sum(t.numel() * t.element_size() for t in outs_host[0]) + gu_host[0].numel() * 2
        s_in, s_cmp, s_out = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
        ev_in = [torch.cuda.Event() for _ in range(NBUF)]
        ev_cmp = [torch.cuda.Event() for _ in range(NBUF)]
        ev_out = [torch.cuda.Event() for _ in range(NBUF)]
        keep = [None] * NBUF

        def e2e_steps(n):
            for i in range(n):
                j = i % NBUF
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_cmp[j])                  # the kernels that read this input buffer are done
                    for d, src in zip(dev_in[j], host):
                        d.copy_(src, non_blocking=True)
                    ev_in[j].record(s_in)
                with torch.cuda.stream(s_cmp):
                    s_cmp.wait_event(ev_in[j])
                    s_cmp.wait_event(ev_out[j])                 # results of step i-NBUF have left the device
                    y, grads = step(*dev_in[j])
                    keep[j] = (y, grads)
                    ev_cmp[j].record(s_cmp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_cmp[j])
                    for dst, src in zip(outs_host[j], [y] + grads[:4]):
                        dst.copy_(src, non_blocking=True)
                    gu_host[j].copy_(grads[4], non_blocking=True)
                    ev_out[j].record(s_out)
            for st in (s_in, s_cmp, s_out):
                torch.cuda.current_stream().wait_stream(st)

        # warm-up: the host<->device copy path of these (virtualised) boxes needs 0.5-2 s of traffic to reach its
        # steady rate; run blocks of 8 steps until two consecutive blocks agree within 4 % (at most 20 blocks)
        prev = None
        for _ in range(20):
            w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0.record()
            e2e_steps(8)
            w1.record()
            torch.cuda.synchronize()
            cur = w0.elapsed_time(w1)
            if world > 1:
                tw = torch.tensor([cur], device=dev, dtype=torch.float64)
                dist.all_reduce(tw, op=dist.ReduceOp.MAX)
                cur = float(tw.item())
            if prev is not None and abs(cur - prev) <= 0.04 * cur:
                break
            prev = cur
        barrier()
        # three consecutive blocks of steps inside one timed region; the per-block times are reported as well,
        # because the host-memory path of a shared box is the one noisy part of this measurement
        kblock = max(2, min(args.steps, 48) // 3)            # the fill and drain of the 3-stage pipeline are inside the timed region
        ksteps = 3 * kblock
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        marks[0].record()
        for i in range(3):
            e2e_steps(kblock)
            marks[i + 1].record()
        barrier()
        a, b_ = marks[0], marks[3]
        ems = a.elapsed_time(b_) / ksteps
        block_ms = [round(marks[i].elapsed_time(marks[i + 1]) / kblock, 3) for i in range(3)]
        if world > 1:
            tms = torch.tensor([ems], device=dev, dtype=torch.float64)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ems = float(tms.item())
        e2e = {"value": world * B * T / (ems * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": ems, "steps": ksteps, "ms_per_step_blocks": block_ms,
               "api": "rwkv_lm_ext_b200.RUN_CUDA_RWKV6 + .backward; pinned host tensors in, all results out, "
                      "copy-in / kernels / copy-out of consecutive steps pipelined on 3 CUDA streams"}

    # ---- BASELINE metric (ii) on every rank (its all_gather is a collective)
    bi = None
    if not args.no_bi_encoder:
        bi = run_bi_encoder(args, M, torch, dist, dev, rank, world, barrier)

    # ---- BASELINE configs[3]: data-parallel LoRA SFT step (fwd + bwd + NCCL gradient all-reduce + AdamW) on every rank
    sft_res = None
    if not args.no_sft:
        sys.path.insert(0, os.path.join(ROOT, "profiles"))
        import bench_sft
        sft_res = {}
        for mode, graphs in (("eager", False), ("cuda_graphs", True)):
            try:
                sft_res[mode], _ = bench_sft.run(layers=24, graphs=graphs, steps_per_bucket=2)
            except Exception as e:      # an extra key must never take the headline measurement down with it
                sft_res[mode] = {"failed": f"{type(e).__name__}: {e}"[:300]}
            barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peak, peak_src = peaks()
    elems = B * T * C
    dom_is_bwd = bwd_ms >= fwd_ms
    dom_ms = bwd_ms if dom_is_bwd else fwd_ms
    dom_bytes = elems * (BYTES_BWD if dom_is_bwd else BYTES_FWD)
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    impl_name = {0: "auto", 1: "simt", 2: "tc"}[M.load().wkv6b200_get_impl()]
    traffic = None
    try:      # dram__bytes_read.sum + dram__bytes_write.sum per launch, from the committed ncu --set full capture
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")))
        traffic = tj["wkv6_tc3_bwd_kernel" if dom_is_bwd else "wkv6_tc3_fwd_kernel"]["dram_bytes_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src,
                "kernel": ("wkv6 backward" if dom_is_bwd else "wkv6 forward") + f" ({impl_name})",
                "algorithmic_bytes_per_launch": dom_bytes, "launch_ms": dom_ms,
                "fwd_ms": fwd_ms, "bwd_ms": bwd_ms,
                # the whole step against the roofline: the 28 B/element of forward + backward over the timed region itself
                # (fwd_ms / bwd_ms come from the split run behind it, whose extra events cost a few microseconds per step)
                "step_frac": elems * (BYTES_FWD + BYTES_BWD) / (ms * 1e-3) / 1e9 / peak}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config(world),
            "clocks": clocks, "gpu_launches": int(launches), "roofline": roofline, "randn_decay": randn_decay}
    line["config"]["launch"] = ("CUDA-graph replay of the captured step (memset + forward kernel + backward kernel)"
                                if graph is not None else "eager (Python-launched) steps")
    line["eager_ms_per_step"] = eager_ms
    if e2e:
        line["e2e"] = e2e
    if bi:
        line["bi_encoder"] = bi
    if sft_res:
        line["sft"] = sft_res

    # ---- the reference's own CUDA kernels on the same inputs (not part of the contract; context)
    try:
        from oracle import ref_cuda
        if world == 1 and ref_cuda.available("wkv6"):
            def ref_step():
                y, ew = ref_cuda.wkv6_forward(r, k, v, w, u)
                return ref_cuda.wkv6_backward(r, k, v, ew, u, gy)
            ref_step()
            torch.cuda.synchronize()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                ref_step()
            b_.record()
            torch.cuda.synchronize()
            rms = a.elapsed_time(b_) / 3
            line["reference_cuda"] = {"value": B * T / (rms * 1e-3), "unit": UNIT, "ms_per_step": rms,
                                      "what": "reference cuda/wkv6_cuda.cu (oracle/_ref) incl. its fp32 ew pre-pass, same GPU"}
    except Exception as e:
        line["reference_cuda"] = {"unavailable": f"{type(e).__name__}: {e}"}

    if world == 1 and not args.no_cpu_baseline:
        val, cores, sec, runs, _ = run_cpu(1000, 1, budget_s=12.0)
        line["cpu_baseline"] = {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": f"fwd+bwd on B={CPU_SAMPLE['B']} T={CPU_SAMPLE['T']} H={CPU_SAMPLE['H']} "
                                          f"(1/8 of one step's batch), mean of {runs} runs of {sec:.2f} s, {cores} threads"}
        # BASELINE configs[0]'s recurrence: the reference's own pure-PyTorch CPU path, unmodified, and this library on the
        # same inputs (bf16) -- a live parity check against the reference's code and the CPU/GPU time of that call
        rp = run_reference_python()
        if rp:
            rr, kk, vv, ww, uu = (t.to(dev).bfloat16().contiguous() for t in rp["_inputs"])
            Br, Tr, Cr = rr.shape
            with torch.no_grad():
                for _ in range(3):
                    yo = M.RUN_CUDA_RWKV6(Br, Tr, Cr, Cr // 64, rr, kk, vv, ww, uu)
                a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a_.record()
                for _ in range(20):
                    yo = M.RUN_CUDA_RWKV6(Br, Tr, Cr, Cr // 64, rr, kk, vv, ww, uu)
                b_.record()
                torch.cuda.synchronize()
            yr = rp["_y"].double()
            info = {k_: v_ for k_, v_ in rp.items() if not k_.startswith("_")}
            info["ours_same_call_ms"] = a_.elapsed_time(b_) / 20
            info["ours_tokens_per_s_forward"] = Br * Tr / (info["ours_same_call_ms"] * 1e-3)
            info["relrms_ours_vs_reference"] = float(((yo.double().cpu() - yr).norm() / yr.norm()).item())
            line["cpu_baseline"]["reference_python"] = info
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
