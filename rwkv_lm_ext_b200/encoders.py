"""Batched, GPU-resident forward of the reference's bi-directional encoder on the fused kernels
(SURVEY.md section 8(f) rank 3).

`bi_encoder_hidden(model, idx)` / `bi_encoder_encode(model, idx)` compute `RwkvEncoder.forward(idx, True)[1]`
and `RwkvEncoder.encode_sentence(idx)` (src/model_encoder_run.py:296-350; the trainer twin is
`src/model_ext.py:398-437`) on any module tree with the reference's attribute names

    emb, blocks[i].{ln0 (i == 0), ln1, ln2, att, ffn}, ln_out, args.emb_id / args.pad_id (or emb_id, pad_id)

Per layer ("semantics 2": a causal pass over the tokens and one over each row's reversed prefix, averaged):

    mask, rev_idx           one kernel on the device (the reference loops over the batch on the host)
    r,k,v,g,w  (x2)         tmix_x060_project: shift-lerp + ddlerp kernels around the cuBLAS Linears
    reverse gathers         128-bit gather kernel
    WKV6 (x2)               tcgen05 / TMA chunked kernel
    GroupNorm * silu(gate)  one kernel
    channel mix             cmix_x060_forward: 3 fused elementwise kernels around the two GEMMs
"""
import torch
import torch.utils.checkpoint

from . import cmix, heads, ops, tmix


def _ids(model):
    a = getattr(model, "args", None)
    emb_id = getattr(a, "emb_id", getattr(model, "emb_id", 1))
    pad_id = getattr(a, "pad_id", getattr(model, "pad_id", 0))
    return int(emb_id), int(pad_id)


def bi_tmix_forward(att, x, rev_idx):
    """bi_att_forward_batch (src/model_encoder_run.py:64-75, :77-93) on the fused kernels."""
    B, T, C = x.shape
    H = att.time_faaaa.shape[0]
    # both directions as ONE batch of 2B rows (the reversed sequences behind the plain ones): every kernel and every
    # Linear of the projection runs once on twice the rows, the recurrence as one launch of 2*B*H streams; the gate is
    # only needed for the plain direction (the reference computes and drops the reversed one)
    xx = heads.stack_reversed(x, rev_idx)
    r, k, v, g, w = tmix.tmix_x060_project(att, xx, gate_rows=B)
    y2 = ops.RUN_CUDA_RWKV6(2 * B, T, C, H, r, k, v, w, att.time_faaaa)
    # y2[:B] plain, y2[B:] still in reversed token order; passed whole, so that its gradient is one [2B,T,C] tensor
    z = heads.groupnorm_gate_pair(y2, None, rev_idx, g, att.ln_x.weight, att.ln_x.bias, H, att.ln_x.eps, gate_act="silu")
    return att.output(z)


def _ffn(ffn, h):
    if all(hasattr(ffn, n) for n in ("time_maa_k", "time_maa_r", "key", "receptance", "value")):
        return cmix.cmix_x060_forward(ffn, h)                         # x060 channel mix on the fused kernels
    return ffn(h)


def blocks_forward(blocks, x, ln_out, att, checkpoint=False):
    """ln_out(block_L(... block_1(x))) for `Block.forward` of src/model.py:904-933 (x = ln0(x) in block 0;
    x = x + att(ln1(x)); x = x + ffn(ln2(x))), with every residual add fused with the LayerNorm that follows it
    (heads.add_layernorm: one pass over the residual stream instead of an add pass and a LayerNorm pass).
    `att(blk, h)` computes the time-mix output of a block from its normalised input.
    checkpoint=True: every block body (x, h) -> (x', h') runs under non-reentrant torch.utils.checkpoint, like the
    reference's trainers (deepspeed.checkpointing.checkpoint(block)); a training step then keeps only the two
    block-boundary tensors of each layer and recomputes the block in the backward."""
    def ln(mod, x_, delta=None):
        return heads.add_layernorm(x_, delta, mod.weight, mod.bias, mod.eps)

    def body(blk, nxt, x_, h_):
        x_, h_ = ln(blk.ln2, x_, att(blk, h_))                        # x += att(ln1(x));  h = ln2(x)
        return ln(nxt, x_, _ffn(blk.ffn, h_))                         # x += ffn(ln2(x));  h = next ln1(x) / ln_out(x)
    h = None
    n = len(blocks)
    for i, blk in enumerate(blocks):
        if i == 0 and hasattr(blk, "ln0"):
            x = ln(blk.ln0, x)[1]
        if h is None:
            h = ln(blk.ln1, x)[1]
        nxt = blocks[i + 1].ln1 if i + 1 < n else ln_out
        if checkpoint and torch.is_grad_enabled():
            x, h = torch.utils.checkpoint.checkpoint(body, blk, nxt, x, h, use_reentrant=False)
        else:
            x, h = body(blk, nxt, x, h)
    return h


def bi_encoder_hidden(model, idx, checkpoint=False):
    """ln_out(blocks(emb(idx)))  [B,T,D] in the model's dtype (bf16 weights expected).  Differentiable on the same
    fused kernels as the inference forward; checkpoint=True recomputes every block in the backward (blocks_forward)."""
    emb_id, pad_id = _ids(model)
    idx = idx.contiguous()
    _, rev_idx = heads.create_mask_and_rev_idx(idx, emb_id, pad_id)
    return blocks_forward(model.blocks, model.emb(idx), model.ln_out, lambda blk, h: bi_tmix_forward(blk.att, h, rev_idx),
                          checkpoint)


def bi_encoder_encode(model, idx, checkpoint=False):
    """encode_sentence: the hidden state at each row's first `emb_id` token.  [B,D]."""
    emb_id, _ = _ids(model)
    hidden = bi_encoder_hidden(model, idx, checkpoint)
    return heads.eos_gather(hidden.contiguous(), idx, emb_id)[0]


# ------------------------------------------------------------------------------------------------
# uni-directional task models (src/model_ext.py:172-212, :1690-1769; src/model_run.py:760-883)
# ------------------------------------------------------------------------------------------------
def _base(wrapper):
    return getattr(wrapper, "rwkvModel", wrapper)


def causal_hidden(model, idx, checkpoint=False):
    """ln_out(blocks(emb(idx)))  [B,T,D] of the plain (causal) RWKV-6 model -- the body shared by
    `RwkvForSequenceEmbedding.forward` (src/model_ext.py:1739-1762) and `RwkvForClassification.forward`
    (src/model_ext.py:183-205) -- with every block on the fused kernels.  Right padding never reaches a position
    before it, so a padded batch gives each row what the reference's one-sentence-at-a-time inference classes
    (src/model_run.py:815-848) compute for it.  checkpoint: recompute every block in the backward (blocks_forward)."""
    base = _base(model)
    return blocks_forward(base.blocks, base.emb(idx.contiguous()), base.ln_out,
                          lambda blk, h: tmix.tmix_x060_forward(blk.att, h), checkpoint)


def sequence_embedding(wrapper, idx, variant="train", checkpoint=False):
    """`RwkvForSequenceEmbedding.forward`: hidden states -> position of the first `embedding_id` token (bit-exact
    index kernel) -> pooling (`weightedmean` / `lasttoken` / `avg`; variant "train" = src/model_ext.py:1708-1738,
    "infer" = src/model_run.py:777-797) -> optional dense + tanh head.  `wrapper` carries the reference's
    attribute names: rwkvModel, embedding_id, pooling_type, add_mlp, dense, activation."""
    emb_id = int(getattr(wrapper, "embedding_id", 1))
    hidden = causal_hidden(wrapper, idx, checkpoint).contiguous()
    pos = heads.eos_index(idx, emb_id)
    x = heads.pooling(hidden, pos, getattr(wrapper, "pooling_type", "weightedmean"), variant)
    if getattr(wrapper, "add_mlp", False):
        x = wrapper.activation(wrapper.dense(x.to(wrapper.dense.weight.dtype)))
    return x


def classification_logits(wrapper, idx, checkpoint=False):
    """`RwkvForClassification.forward` (src/model_ext.py:183-211): score(hidden)[b, first class_id token].  The row is
    gathered BEFORE the score Linear (same numbers, T times fewer FLOPs than scoring every token).  This is also the
    reference's cross-encoder: rows are "query [sep] document [cls]" (see `cross_encoder_rows`)."""
    cls_id = int(getattr(wrapper, "class_id", 1))
    hidden = causal_hidden(wrapper, idx, checkpoint).contiguous()
    row, _ = heads.eos_gather(hidden, idx, cls_id)
    return wrapper.score(row.to(wrapper.score.weight.dtype))


def cross_encoder_rows(queries, documents, max_len, sep_id=2, class_id=1, pad_id=0):
    """Token rows of the cross-encoder (peft_train/data_collators.py / data/custom_datasets.py
    `cross_encoder_pad_and_truncated_according_data`): query + [sep] + document, truncated to max_len - 1, then the
    class token, right-padded.  queries / documents: lists of token-id lists.  Returns int64 [B, max_len] (CPU)."""
    rows = []
    for q, d in zip(queries, documents):
        ids = (list(q) + [sep_id] + list(d))[: max_len - 1] + [class_id]
        rows.append(ids + [pad_id] * (max_len - len(ids)))
    return torch.tensor(rows, dtype=torch.long)


def length_buckets(lengths, max_tokens, multiple=64):
    """Batches of sequence indices for a corpus of ragged sequences: sorted by length, each batch padded to its longest
    member (rounded up to `multiple`) with at most `max_tokens` padded tokens -- the batched, GPU-resident replacement
    of the reference's one-sentence-at-a-time loops (tests/TestBiEncoder.py:22-36, src/model_run.py:954-968)."""
    order = sorted(range(len(lengths)), key=lambda i: lengths[i])
    batches, cur, width = [], [], 0
    for i in order:
        w = -(-max(1, lengths[i]) // multiple) * multiple
        if cur and max(width, w) * (len(cur) + 1) > max_tokens:
            batches.append((cur, width))
            cur, width = [], 0
        cur.append(i)
        width = max(width, w)
    if cur:
        batches.append((cur, width))
    return batches


def encode_corpus(model, sequences, fn=None, max_tokens=32768, end_id=1, pad_id=0):
    """Embeds (or scores) a list of token-id lists of any lengths.  Each sequence gets `end_id` appended if it does not
    end with it; batches come from `length_buckets`; `fn(model, idx)` defaults to `bi_encoder_encode` for a bare
    encoder and `sequence_embedding` for a wrapper with `rwkvModel`.  Results are returned in input order."""
    if fn is None:
        fn = sequence_embedding if hasattr(model, "rwkvModel") else bi_encoder_encode
    seqs = [list(s) if len(s) and s[-1] == end_id else list(s) + [end_id] for s in sequences]
    dev = next(model.parameters()).device
    out = [None] * len(seqs)
    for members, width in length_buckets([len(s) for s in seqs], max_tokens):
        idx = torch.full((len(members), width), pad_id, dtype=torch.long)
        for r, i in enumerate(members):
            idx[r, : len(seqs[i])] = torch.tensor(seqs[i], dtype=torch.long)
        res = fn(model, idx.to(dev, non_blocking=True))
        for r, i in enumerate(members):
            out[i] = res[r]
    return torch.stack(out)


class GraphedForward:
    """`fn(model, idx)` for ONE input shape as a CUDA-graph replay: the forwards above make ~130 launches per layer, a
    third of them a few microseconds long, and launched eagerly the GPU waits for the host between them (1B6 bi-encoder,
    64 x 512 tokens: ~10 % of the step).  Every kernel of the path takes its scratch from torch's allocator or from
    stream-ordered allocations and nothing synchronises with the host, so the whole forward captures.

        enc = GraphedForward(bi_encoder_encode, model, idx)      # warms up, captures
        emb = enc(idx2)                                          # idx2.shape == idx.shape; emb is overwritten by the next call

    Inference only (captured under no_grad).  Parameters are read in place: weight updates are seen by later replays."""

    def __init__(self, fn, model, example_idx, warmup=2):
        assert example_idx.is_cuda
        self.fn, self.model = fn, model
        self.static_idx = example_idx.clone()
        side = torch.cuda.Stream(device=example_idx.device)
        side.wait_stream(torch.cuda.current_stream(example_idx.device))
        with torch.cuda.stream(side), torch.no_grad():
            for _ in range(warmup):
                fn(model, self.static_idx)
        torch.cuda.current_stream(example_idx.device).wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.no_grad(), torch.cuda.graph(self.graph):
            self.static_out = fn(model, self.static_idx)

    def __call__(self, idx):
        assert idx.shape == self.static_idx.shape and idx.dtype == self.static_idx.dtype, "one graph per input shape"
        self.static_idx.copy_(idx, non_blocking=True)
        self.graph.replay()
        return self.static_out
