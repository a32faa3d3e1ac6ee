"""Host-side logic of the data-parallel SFT path on CPU (BASELINE.json configs[3]): the bucketed batch sampler against
index sequences produced by the REFERENCE's MyBatchSampler (tests/golden/make_sampler_golden.py), the LoRA / PiSSA
linear against the reference formulas, the adapter checkpoint format, and -- world_size 2, gloo -- that the bucketed
asynchronous gradient all-reduce gives every rank the gradient of the full batch."""
import json
import math
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from rwkv_lm_ext_b200 import sft

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sampler_golden.json")


def test_bucket_sampler_matches_the_reference():
    gold = json.load(open(GOLDEN))
    for c in gold["sampler"]:
        for rank, ref in enumerate(c["ranks"]):
            s = sft.BucketBatchSampler(c["cumulative_sizes"], c["batch_sizes"], rank, c["world"], c["skipped"])
            assert [list(b) for b in s] == ref["batches"], (c, rank)
            assert len(s) == ref["len"]
    col = gold["collate"]
    ids, lab = sft.pad_only_according_data(col["features"])
    assert ids.tolist() == col["input_ids"] and lab.tolist() == col["labels"]


def test_bucket_sampler_ranks_are_disjoint_and_in_one_bucket():
    lengths = [64, 128, 256, 512, 1024, 2048]
    bss = sft.bucket_batch_sizes(lengths)                      # README.md:80
    assert bss == [32, 16, 8, 4, 2, 1]
    ds = sft.SyntheticSftBuckets(lengths, per_bucket=64, vocab=1000)
    world = 2
    its = [iter(sft.BucketBatchSampler(ds.cumulative_sizes, bss, r, world)) for r in range(world)]
    seen = set()
    for step, batches in enumerate(zip(*its)):
        buckets = {its_ and sft.BucketBatchSampler(ds.cumulative_sizes, bss).bucket_of(i) for b in batches for i in b for its_ in [1]}
        assert len(buckets) == 1                               # every rank works on the same length bucket in a step
        flat = [i for b in batches for i in b]
        assert not (set(flat) & seen) and len(set(flat)) == len(flat)
        seen.update(flat)
        b0 = buckets.pop()
        assert all(len(b) == bss[b0] for b in batches)
        feats = [ds[i] for i in batches[0]]
        ids, lab = sft.pad_only_according_data(feats)
        assert ids.shape == lab.shape == (bss[b0], lengths[b0])
        assert (lab[:, 0] == -100).all() or lengths[b0] <= 2
    assert step + 1 == sum(64 // (b * world) for b in bss)


def test_lora_linear_matches_the_reference_formulas():
    torch.manual_seed(0)
    m = sft.LoraLinear(24, 16, r=4, alpha=32)
    with torch.no_grad():
        m.lora_B.normal_()
    x = torch.randn(5, 24)
    ref = F.linear(x, m.weight) + (32 / 4) * F.linear(F.linear(x, m.lora_A), m.lora_B)     # src/rwkvLinear.py:94-96
    assert torch.allclose(m(x), ref)
    w0 = m.weight.data.clone()
    m.pissa_init(svd_niter=8)                                                              # src/rwkvLinear.py:66-75
    assert torch.allclose(m.weight.data + m.lora_B.data @ m.lora_A.data, w0, atol=1e-5)
    assert torch.allclose(m(x), F.linear(x, w0), atol=1e-4)                               # the decomposition is exact at init
    S = torch.linalg.svdvals(w0)                              # svd_lowrank is randomised: near the best rank-4 energy
    assert (m.lora_B.data @ m.lora_A.data).norm() >= 0.9 * S[:4].norm()


def test_lora_linear_fused_backward_equals_the_eager_chain():
    """_LoraFn folds the scaling and both additions into the GEMMs; with a GradBuckets buffer the adapter gradients are
    accumulated in place (no tensor returned to autograd) and the bucket bookkeeping is told."""
    torch.manual_seed(3)
    for pissa in (False, True):
        m = sft.LoraLinear(24, 16, r=4, alpha=32).double()
        m.pissa = pissa
        with torch.no_grad():
            m.lora_B.normal_()
        x = torch.randn(3, 5, 24, dtype=torch.float64, requires_grad=True)
        gy = torch.randn(3, 5, 16, dtype=torch.float64)
        s = 1.0 if pissa else 32 / 4
        ref = F.linear(x, m.weight) + s * F.linear(F.linear(x, m.lora_A), m.lora_B)
        want = torch.autograd.grad(ref, (x, m.weight, m.lora_A, m.lora_B), gy)
        out = m(x)
        assert out.shape == ref.shape and torch.allclose(out, ref, atol=1e-12)
        got = torch.autograd.grad(out, (x, m.weight, m.lora_A, m.lora_B), gy)
        for a, b in zip(got, want):
            assert torch.allclose(a, b, atol=1e-10)
        # frozen weight, gradients straight into the flat buffer: two backward passes accumulate, the hooks fire once each
        m.weight.requires_grad = False
        sinks_before = dict(sft._GRAD_SINKS)   # SftTrainer never calls GradBuckets.remove(): earlier tests' trainers keep theirs
        gbk = sft.GradBuckets([m.lora_A, m.lora_B], n_buckets=1)
        try:
            for rep in (1, 2):
                m(x).backward(gy)
                assert gbk._pending == [0]
                gbk._pending, gbk._seen = [2], set()           # what finish() does, without dividing
                assert torch.allclose(m.lora_A.grad, rep * want[2], atol=1e-10) and torch.allclose(m.lora_B.grad, rep * want[3], atol=1e-10)
                assert m.lora_A.grad.data_ptr() >= gbk.flat.data_ptr()                  # still views of the flat buffer
            assert torch.allclose(x.grad, 2 * want[0], atol=1e-10) and m.weight.grad is None
        finally:
            gbk.remove()
        assert sft._GRAD_SINKS == sinks_before
        m.train()
        m.lora_dropout.p = 0.5                                   # dropout: the eager chain (different mask per call)
        assert m(x).shape == ref.shape


def test_trainable_checkpoint_format(tmp_path):
    model = sft.RwkvSft(layers=1, D=64, H=1, ffn=96, vocab=50, lora_r=2, lora_alpha=4)
    train = model.mark_trainable()
    names = [n for n, p in model.named_parameters() if p.requires_grad]
    assert names and all("lora_" in n for n in names) and len(train) == len(names) == 16       # 8 Linears x (A, B)
    path = sft.save_trainable(model, str(tmp_path), "/somewhere/RWKV-x060-World-1B6.pth")
    assert os.path.basename(path) == "RWKV-x060-World-1B6.pth.pth"                           # peft_train/Callbacks.py:24
    sd = torch.load(path)
    assert sorted(sd) == sorted(names)
    assert "blocks.0.att.receptance.lora_A" in sd and "blocks.0.ffn.value.lora_B" in sd      # the reference's names
    other = sft.RwkvSft(layers=1, D=64, H=1, ffn=96, vocab=50, lora_r=2, lora_alpha=4)
    info = sft.load_trainable(other, path)
    assert not info.unexpected_keys
    assert torch.equal(other.blocks[0].att.key.lora_A, model.blocks[0].att.key.lora_A)
    init = sft.pissa_init_all(model, svd_niter=2, init_file=str(tmp_path / "init_pissa.pth"))
    assert "blocks.0.att.key.init_lora_A" in init and os.path.exists(tmp_path / "init_pissa.pth")   # peft_train_sft.py:195-196
    state = sft.RwkvSft(layers=1, D=64, H=1, ffn=96, vocab=50, train_type="state")
    state.mark_trainable()
    assert [n for n, p in state.named_parameters() if p.requires_grad] == ["blocks.0.att.time_state"]


class _Tiny(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.a = sft.LoraLinear(12, 20, r=3, alpha=6)
        self.b = sft.LoraLinear(20, 7, r=3, alpha=6)

    def forward(self, x):
        return self.b(torch.tanh(self.a(x)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _dp_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(1)
        model = _Tiny()
        with torch.no_grad():
            model.a.lora_B.normal_()
            model.b.lora_B.normal_()
        for n, p in model.named_parameters():
            p.requires_grad = "lora_" in n
        params = [p for p in model.parameters() if p.requires_grad]
        gb = sft.GradBuckets(params, n_buckets=3)
        assert len(gb.buckets) >= 2
        x, y = torch.randn(8, 12, generator=torch.Generator().manual_seed(2)), torch.randn(8, 7, generator=torch.Generator().manual_seed(3))
        for it in range(2):                                    # twice: the bucket bookkeeping must reset
            lo = rank * 4
            loss = F.mse_loss(model(x[lo:lo + 4]), y[lo:lo + 4])
            loss.backward()
            flat = gb.finish().clone()
            if it == 0:
                gb.zero()
        if rank == 0:
            torch.save({"flat": flat, "names": [n for n, p in model.named_parameters() if p.requires_grad],
                        "grads": {n: p.grad.clone() for n, p in model.named_parameters() if p.requires_grad}}, out)
    finally:
        dist.destroy_process_group()


def test_two_rank_bucketed_allreduce_equals_full_batch_gradient(tmp_path):
    out = str(tmp_path / "g.pt")
    mp.spawn(_dp_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = torch.load(out)
    torch.manual_seed(1)
    model = _Tiny()
    with torch.no_grad():
        model.a.lora_B.normal_()
        model.b.lora_B.normal_()
    x, y = torch.randn(8, 12, generator=torch.Generator().manual_seed(2)), torch.randn(8, 7, generator=torch.Generator().manual_seed(3))
    F.mse_loss(model(x), y).backward()                        # one process, the whole batch
    for n, p in model.named_parameters():
        if "lora_" in n:
            assert torch.allclose(got["grads"][n], p.grad, atol=1e-6), n


def test_sft_loss_ignores_masked_labels_and_pulls_the_max_logit():
    torch.manual_seed(0)
    logits = torch.randn(2, 5, 11, requires_grad=True)
    tgt = torch.randint(0, 11, (2, 5))
    tgt[0, :2] = -100
    loss = sft.sft_loss(logits, tgt)
    ref = F.cross_entropy(logits.detach().view(-1, 11)[tgt.view(-1) != -100], tgt.view(-1)[tgt.view(-1) != -100])
    assert math.isclose(loss.item(), ref.item(), rel_tol=1e-6)
    loss.backward()
    plain = torch.autograd.grad(F.cross_entropy(logits.view(-1, 11), tgt.view(-1)), logits)[0]
    extra = logits.grad - plain                                # L2Wrap: 1e-4 / (B*T) * max logit at its position
    mx, ids = logits.detach().max(-1, keepdim=True)
    want = torch.zeros_like(extra).scatter_(-1, ids, mx * 1e-4 / 10)
    assert torch.allclose(extra, want, atol=1e-7)
