"""One process per GPU (torch.distributed, NCCL over NVLink/NVSwitch): data-parallel gradient all-reduce through one
flat bucket, and the vocab-shard / top-k exchange helpers.  The reference has no counterpart (only nn.DataParallel,
NN/trainers/base.py:32-34); the contract is "N ranks == 1 rank on the same global batch" (SURVEY.md 8e)."""
from __future__ import annotations

from typing import List, Sequence, Tuple

import torch
import torch.distributed as dist

from . import lib as L
from .lib import check, ptr, stream, count_launches


def shard_range(n_rows: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous row block [begin, end) of a table row-sharded over `world` ranks (ceil(n/world) rows each)."""
    per = (n_rows + world - 1) // world
    b = min(rank * per, n_rows)
    return b, min(b + per, n_rows)


def split_batch(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Rows of a global batch owned by `rank` (strong scaling: the global batch is fixed)."""
    return shard_range(n, rank, world)


def bucket_layout(sizes: Sequence[int], align: int = 4) -> Tuple[List[int], int]:
    """Element offsets of each tensor inside the flat bucket (each start aligned to `align` elements) and total size."""
    offs, o = [], 0
    for n in sizes:
        offs.append(o)
        o += (n + align - 1) // align * align
    return offs, o


def chunk_map(sizes: Sequence[int]) -> torch.Tensor:
    rows = [(ti, ci) for ti, n in enumerate(sizes) for ci in range((n + L.ADAM_CHUNK - 1) // L.ADAM_CHUNK)]
    return torch.tensor(rows, dtype=torch.int32).reshape(-1, 2)


class GradSync:
    """Averages the gradients of `params` over all ranks: pack -> ONE all-reduce of a flat fp32 bucket -> unpack."""

    def __init__(self, params, group=None):
        self.params = [p for p in params if p.requires_grad]
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.sizes = [p.numel() for p in self.params]
        self.offsets, self.total = bucket_layout(self.sizes)
        dev = self.params[0].device
        self.bucket = torch.zeros(self.total, device=dev, dtype=torch.float32)
        self.cmap = chunk_map(self.sizes).to(dev)

    def allreduce_bucket(self):
        if self.world > 1:
            dist.all_reduce(self.bucket, op=dist.ReduceOp.SUM, group=self.group)

    def _table(self):
        rows = []
        for p, n, o in zip(self.params, self.sizes, self.offsets):
            if p.grad is None:
                p.grad = torch.zeros_like(p)
            g = p.grad if p.grad.is_contiguous() else p.grad.contiguous()
            p.grad = g
            rows.append((g.data_ptr(), n, o))
        # gradient buffers keep their addresses from step to step: the device copy of the table is reused (a pageable
        # host->device copy every step would block the host until the stream has drained)
        key = tuple(r[0] for r in rows)
        if getattr(self, "_tab_key", None) != key:
            if torch.cuda.is_current_stream_capturing():  # see FusedAdam._tables: staged through pre-allocated pinned memory
                pinned, devbuf = self._capture_bufs
                pinned.copy_(torch.tensor(rows, dtype=torch.int64))
                devbuf.copy_(pinned, non_blocking=True)
                self._tab = devbuf
            else:
                self._tab = torch.tensor(rows, dtype=torch.int64).to(self.bucket.device)
            self._tab_key = key
        return self._tab

    def prepare_capture(self):
        """Buffers for the gradient-address table, allocated before a CUDA-graph capture."""
        n = len(self.params)
        self._capture_bufs = (torch.empty(n, 3, dtype=torch.int64).pin_memory(), torch.empty(n, 3, dtype=torch.int64, device=self.bucket.device))
        self._tab_key = None

    def pack(self):
        """Gradients -> flat bucket, scaled by 1/world (one launch)."""
        tab = self._table()
        check(L.load().rbm_bucket_pack(ptr(tab), ptr(self.cmap), self.cmap.shape[0], ptr(self.bucket), 1.0 / self.world, 0, stream()),
              "bucket_pack")
        count_launches()

    def unpack(self):
        """Flat bucket -> gradients (one launch)."""
        tab = self._table()
        check(L.load().rbm_bucket_pack(ptr(tab), ptr(self.cmap), self.cmap.shape[0], ptr(self.bucket), 1.0, 1, stream()), "bucket_unpack")
        count_launches()

    def allreduce_grads(self):
        if self.world == 1:
            return
        self.pack()
        self.allreduce_bucket()
        self.unpack()


def gather_topk(vals: torch.Tensor, ids: torch.Tensor, group=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """All-gather per-shard top-k lists [U,k] -> [S,U,k] (80 B per user per shard for k=10)."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return vals.unsqueeze(0), ids.unsqueeze(0)
    vs = [torch.empty_like(vals) for _ in range(world)]
    is_ = [torch.empty_like(ids) for _ in range(world)]
    dist.all_gather(vs, vals.contiguous(), group=group)
    dist.all_gather(is_, ids.contiguous(), group=group)
    return torch.stack(vs), torch.stack(is_)


def sharded_full_catalogue_topk(last_hidden: torch.Tensor, table: torch.Tensor, bias, num_items: int, k: int, group=None,
                                exclude=None):
    """Vocab-parallel top-k: every rank scores ALL users against ITS row block of the (replicated or locally held)
    table with global item ids, the per-shard lists are exchanged and merged with the same (score desc, id asc) rule,
    so the result does not depend on the number of shards.  ``exclude`` ([U, n] global item ids, see ``ops.score_topk``):
    the users are the same on every rank, so every shard filters with the same rows."""
    from . import ops
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    b, e = shard_range(num_items, rank, world)  # items are rows 1..V
    if e > b:
        vals, ids = ops.score_topk(last_hidden, table, bias, 1 + b, 1 + e, k, exclude=exclude)
    else:
        U = last_hidden.shape[0]
        vals = torch.full((U, k), float("-inf"), device=last_hidden.device)
        ids = torch.full((U, k), -1, device=last_hidden.device, dtype=torch.int64)
    gv, gi = gather_topk(vals, ids, group)
    return ops.topk_merge(gv, gi)


# ------------------------------------------------------------------------------------ vocab-parallel cross-entropy
def combine_shard_lse(lse_all: torch.Tensor, loss_all: torch.Tensor, count: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Global log-sum-exp and loss from per-shard CE results (SURVEY.md 8e, BERT CE): ``lse_all [S, cap]`` are the
    per-shard log-sum-exps of the first ``count`` (compacted, masked) rows, ``loss_all [S]`` the per-shard values of
    ``mean(lse_s - target logit if the target lies in shard s else lse_s)`` as ``rbm_ce_fwd`` returns them for a shard.
    Returns (LSE [cap] fp32, loss scalar).  Since a target lies in exactly one shard,
    ``sum_r target_logit[r] = sum_s (sum_r lse_s[r] - count * loss_s)``."""
    S, cap = lse_all.shape
    live = torch.arange(cap, device=lse_all.device) < count.reshape(())
    cnt = count.reshape(()).to(torch.float64)
    # entries beyond `count` are uninitialised memory (possibly inf / nan): select, never multiply
    lse64 = torch.where(live.unsqueeze(0), lse_all.to(torch.float64), torch.zeros((), dtype=torch.float64, device=lse_all.device))
    LSE = torch.logsumexp(lse64, dim=0)
    tgt_sum = (lse64.sum(dim=1) - cnt * loss_all.to(torch.float64)).sum()
    loss = (torch.where(live, LSE, torch.zeros_like(LSE)).sum() - tgt_sum) / cnt
    return LSE.to(torch.float32), loss.to(torch.float32)


class VocabParallelCEFn(torch.autograd.Function):
    """Masked cross-entropy with the output layer row-sharded over the ranks of `group` (SURVEY.md 8e):
    every rank holds the SAME hidden rows and labels and its own block ``w[v_begin:v_end]``, ``bias[v_begin:v_end]``.
    Forward: fused scoring + online softmax against the local block (``rbm_ce_fwd``, targets shifted by ``-v_begin`` so
    that a target outside the block matches no column), all-gather of the per-row log-sum-exps and the shard losses
    ((1 + cap) floats per rank), combination into the global LSE / loss.  Backward: ``rbm_ce_bwd`` with the GLOBAL LSE
    yields this block's dW / db and this block's share of dH; the dH shares are summed with one all-reduce."""

    @staticmethod
    def forward(ctx, hidden, labels, w_shard, bias_shard, v_begin, group, own_rows=None):
        from . import ops
        lib = L.load()
        L.require_cuda(hidden, labels, w_shard, bias_shard)
        ctx.own_rows = own_rows
        h2 = hidden.reshape(-1, hidden.shape[-1]).contiguous()
        n, d = h2.shape
        V1 = w_shard.shape[0]
        labels = labels.reshape(-1).contiguous()
        dev = hidden.device
        rows = torch.empty(n, device=dev, dtype=torch.int32)
        tgt = torch.empty(n, device=dev, dtype=torch.int64)
        count = torch.empty(1, device=dev, dtype=torch.int32)
        nb = lib.rbm_compact_ws_bytes(n)
        ws = ops._ws("compact", nb, dev)
        check(lib.rbm_compact_labels(ptr(labels), n, ptr(rows), ptr(tgt), ptr(count), ptr(ws), nb, stream()), "compact_labels")
        tgt_local = (tgt - int(v_begin)).contiguous()
        lse_s = torch.empty(n, device=dev, dtype=torch.float32)
        loss_s = torch.empty(1, device=dev, dtype=torch.float32)
        nb = lib.rbm_ce_ws_bytes(n, V1, d)
        ws = ops._ws("ce", nb, dev)
        w_shard = w_shard.contiguous()
        check(lib.rbm_ce_fwd(ptr(h2), ptr(rows), ptr(tgt_local), ptr(count), ptr(w_shard), ptr(bias_shard), ptr(lse_s), ptr(loss_s), n, V1,
                             d, ptr(ws), nb, stream()), "ce_fwd")
        count_launches(5)
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        if world > 1:
            lse_list = [torch.empty_like(lse_s) for _ in range(world)]
            loss_list = [torch.empty_like(loss_s) for _ in range(world)]
            dist.all_gather(lse_list, lse_s, group=group)
            dist.all_gather(loss_list, loss_s, group=group)
            lse_all, loss_all = torch.stack(lse_list), torch.cat(loss_list)
        else:
            lse_all, loss_all = lse_s.unsqueeze(0), loss_s
        LSE, loss = combine_shard_lse(lse_all, loss_all, count)
        ctx.save_for_backward(h2, rows, tgt_local, count, w_shard, bias_shard, LSE.contiguous())
        ctx.shape, ctx.group, ctx.world = hidden.shape, group, world
        return loss

    @staticmethod
    def backward(ctx, dloss):
        from . import ops
        lib = L.load()
        h2, rows, tgt_local, count, w_shard, bias_shard, LSE = ctx.saved_tensors
        n, d = h2.shape
        V1 = w_shard.shape[0]
        dloss = dloss.reshape(1).contiguous().float()
        dh = torch.zeros_like(h2)
        dw = torch.empty_like(w_shard)
        db = torch.empty(V1, device=h2.device, dtype=torch.float32)
        nb = lib.rbm_ce_ws_bytes(n, V1, d)
        ws = ops._ws("ce", nb, h2.device)
        check(lib.rbm_ce_bwd(ptr(h2), ptr(rows), ptr(tgt_local), ptr(count), ptr(w_shard), ptr(bias_shard), ptr(LSE), ptr(dloss), ptr(dh),
                             ptr(dw), ptr(db), n, V1, d, ptr(ws), nb, stream()), "ce_bwd")
        count_launches(4)
        if ctx.world > 1:
            if ctx.own_rows is not None and n == ctx.world * ctx.own_rows:
                # the rows are the ranks' slot blocks in rank order and each rank only needs the gradient of ITS block
                # (hybrid_vocab_parallel_loss): reduce-scatter moves half the bytes of an all-reduce
                mine = torch.empty(ctx.own_rows, d, device=dh.device, dtype=dh.dtype)
                dist.reduce_scatter_tensor(mine, dh, op=dist.ReduceOp.SUM, group=ctx.group)
                r = dist.get_rank(ctx.group)
                dh.zero_()
                dh[r * ctx.own_rows:(r + 1) * ctx.own_rows] = mine
            else:
                dist.all_reduce(dh, op=dist.ReduceOp.SUM, group=ctx.group)  # every rank needs the full dH of the replicated rows
        return dh.view(ctx.shape), None, dw, db, None, None, None


def vocab_parallel_cross_entropy(hidden, labels, w_shard, bias_shard, v_begin: int, group=None, own_rows=None):
    """See VocabParallelCEFn.  ``v_begin`` = first row of the output layer held by this rank (``shard_range(V + 1, rank, world)``).
    ``own_rows``: the rows are ``world`` blocks of that many rows in rank order and this rank only consumes the gradient of its own
    block (the backward then reduce-scatters the dH shares instead of all-reducing them; the other blocks' gradient reads as zero)."""
    return VocabParallelCEFn.apply(hidden, labels, w_shard, bias_shard, v_begin, group, own_rows)


# ------------------------------------------------------------ data-parallel batch x vocab-parallel output layer (cfg4)
def masked_row_slots(count: torch.Tensor, rows: torch.Tensor, tgt: torch.Tensor, capacity: int):
    """Fixed-capacity view of a rank's compacted masked rows (``rbm_compact_labels`` output: ``rows[:count]`` are the row ids
    with label != 0, ``tgt[:count]`` their labels; entries beyond ``count`` are uninitialised).  Returns
    ``(live [cap] bool, rows_c [cap] int64, labels_c [cap] int64, overflow 0-dim bool)``: dead slots point at row 0 and carry
    label 0 (= ignored by the cross-entropy), ``overflow`` says that ``count > capacity`` (rows would be dropped)."""
    cap = int(capacity)
    cnt = count.reshape(()).to(torch.int64)
    live = torch.arange(cap, device=rows.device) < cnt
    zero = torch.zeros((), dtype=torch.int64, device=rows.device)
    rows_c = torch.where(live, rows[:cap].to(torch.int64), zero)
    labels_c = torch.where(live, tgt[:cap].to(torch.int64), zero)
    return live, rows_c, labels_c, cnt > cap


def gather_slots(h2: torch.Tensor, live, rows_c, labels_c, group=None):
    """Rows of ``h2`` named by the slots (dead slots zeroed) and their labels, all-gathered over the ranks in rank order:
    ``([world * cap, d], [world * cap])``."""
    slots = h2.index_select(0, rows_c) * live.unsqueeze(1).to(h2.dtype)
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    if world == 1:
        return slots, labels_c
    hs = [torch.empty_like(slots) for _ in range(world)]
    ls = [torch.empty_like(labels_c) for _ in range(world)]
    dist.all_gather(hs, slots.contiguous(), group=group)
    dist.all_gather(ls, labels_c.contiguous(), group=group)
    return torch.cat(hs), torch.cat(ls)


def scatter_slot_grads(dh_all: torch.Tensor, rows_c, live, n: int, cap: int, rank: int, scale: float):
    """This rank's slice of the gathered rows' gradient back onto its ``n`` local rows (times ``scale``)."""
    mine = dh_all[rank * cap:(rank + 1) * cap] * (live.unsqueeze(1).to(dh_all.dtype) * scale)
    dh = torch.zeros(n, dh_all.shape[1], device=dh_all.device, dtype=dh_all.dtype)
    dh.index_add_(0, rows_c, mine)  # live slots hold distinct rows; dead slots add exact zeros to row 0: order-independent
    return dh


class GatherMaskedRowsFn(torch.autograd.Function):
    """SURVEY.md 8(e), BERT CE at cfg4: every rank holds ITS OWN sequences (data parallel); only the rows with a label
    (about 15 %) take part in the vocab-parallel scoring.  Forward: compact the local masked rows on the device
    (``rbm_compact_labels``), place them in ``capacity`` slots (no host sync: the slot count is static, dead slots carry
    label 0), all-gather slots and labels -> ``[world * capacity, d]`` replicated rows for ``vocab_parallel_cross_entropy``.
    Backward: this rank's slice of the (already shard-summed) dH goes back to its local rows, times ``grad_scale``."""

    @staticmethod
    def forward(ctx, hidden, labels, capacity, group, grad_scale):
        from . import ops
        lib = L.load()
        L.require_cuda(hidden, labels)
        h2 = hidden.reshape(-1, hidden.shape[-1])
        n, d = h2.shape
        lab = labels.reshape(-1).contiguous()
        dev = hidden.device
        rows = torch.empty(n, device=dev, dtype=torch.int32)
        tgt = torch.empty(n, device=dev, dtype=torch.int64)
        count = torch.empty(1, device=dev, dtype=torch.int32)
        nb = lib.rbm_compact_ws_bytes(n)
        ws = ops._ws("compact", nb, dev)
        check(lib.rbm_compact_labels(ptr(lab), n, ptr(rows), ptr(tgt), ptr(count), ptr(ws), nb, stream()), "compact_labels")
        count_launches(3)
        cap = n if capacity is None else min(int(capacity), n)
        live, rows_c, labels_c, overflow = masked_row_slots(count, rows, tgt, cap)
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        h_all, l_all = gather_slots(h2, live, rows_c, labels_c, group)
        ctx.save_for_backward(rows_c, live)
        ctx.meta = (hidden.shape, n, d, cap, rank, float(grad_scale))
        ctx.mark_non_differentiable(l_all, overflow)
        return h_all, l_all, overflow

    @staticmethod
    def backward(ctx, dh_all, _dl, _do):
        rows_c, live = ctx.saved_tensors
        shape, n, d, cap, rank, scale = ctx.meta
        return scatter_slot_grads(dh_all, rows_c, live, n, cap, rank, scale).view(shape), None, None, None, None


def hybrid_vocab_parallel_loss(hidden, labels, w_shard, bias_shard, v_begin: int, capacity=None, group=None,
                               compensate_grad_average: bool = True):
    """Masked cross-entropy of the GLOBAL batch when sequences are data-parallel and the output layer is row-sharded
    (BASELINE configs[3]; SURVEY.md 8e).  ``hidden [B_local, L, d]`` / ``labels [B_local, L]`` are this rank's own; returns
    ``(loss, overflow)``: the mean over all labelled positions of all ranks (what one GPU computes on the concatenated batch,
    NN/trainers/bert.py:30-41), and a device flag that is true if some rank had more than ``capacity`` labelled rows
    (``capacity=None``: B_local*L slots, never overflows; about 0.2*B_local*L keeps the exchange at the 15 % mask rate).
    Gradients: ``w_shard`` / ``bias_shard`` get the exact global-batch gradient of their rows (keep them OUT of the
    data-parallel bucket); ``hidden`` gets the global-batch gradient of its rows, multiplied by the world size when
    ``compensate_grad_average`` so that ``GradSync``'s averaging of the body gradients yields the global-batch gradient."""
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    scale = float(world) if compensate_grad_average else 1.0
    h_all, l_all, overflow = GatherMaskedRowsFn.apply(hidden, labels, capacity, group, scale)
    return vocab_parallel_cross_entropy(h_all, l_all, w_shard, bias_shard, v_begin, group, own_rows=h_all.shape[0] // world), overflow


# ------------------------------------------------------------------------ row-sharded item table: input lookup (SURVEY 8e)
def shard_keys(tok_all: torch.Tensor, v_begin: int, v_end: int, padding_idx: int = 0) -> torch.Tensor:
    """Scatter keys of a shard: ``tok - v_begin`` for the tokens this shard owns, ``v_end - v_begin`` (one past the last local
    row = the key ``rbm_scatter_add_sorted`` is told to skip) for everything else, the padding id included."""
    own = (tok_all >= v_begin) & (tok_all < v_end) & (tok_all != padding_idx)
    return torch.where(own, tok_all - v_begin, torch.full_like(tok_all, v_end - v_begin))


class ShardedEmbedFn(torch.autograd.Function):
    """Embedding stage (gather x scale + positions + dropout + pad zeroing) with the item table ROW-SHARDED over the ranks and the
    sequences data-parallel.  Forward: all-gather the token ids (8 B per token), every rank runs the fused kernel on ALL tokens
    against its block -- tokens of other blocks give exact zeros -- and a reduce-scatter hands every rank the rows of its own
    sequences; exactly one addend per element is non-zero, so the result equals the unsharded kernel on the concatenated batch
    bit for bit.  Backward: the rank masks its gradient rows (dropout / padding, global element indices) and reduces ``dpos`` over
    its batch, the rows are all-gathered, and each rank sort/segment-reduces the rows of ITS items into the gradient of its
    block (fixed order = global batch order).  ``grad_unscale``: divide the table gradient by this (the world size when the
    loss pre-multiplies body gradients to compensate ``GradSync``'s averaging; sharded tensors are not averaged)."""

    @staticmethod
    def forward(ctx, tok, table_shard, pos, v_begin, vocab, scale, zero_pad, p, seed, site, group, grad_unscale):
        from . import ops
        lib = L.load()
        L.require_cuda(tok, table_shard, pos)
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        rank = dist.get_rank(group) if dist.is_initialized() else 0
        Bsz, Ln = tok.shape
        d = table_shard.shape[1]
        v_end = int(v_begin) + table_shard.shape[0]
        tok = tok.contiguous()
        if world > 1:
            tok_all = torch.empty(world * Bsz, Ln, device=tok.device, dtype=tok.dtype)
            dist.all_gather_into_tensor(tok_all, tok, group=group)
        else:
            tok_all = tok
        part = torch.empty(world * Bsz, Ln, d, device=tok.device, dtype=torch.float32)
        check(lib.rbm_embed_fwd_shard(ptr(tok_all), ptr(table_shard), ptr(pos), ptr(part), world * Bsz * Ln, Ln, d, int(vocab), int(v_begin),
                                      v_end, float(scale), int(zero_pad), float(p), seed, site, stream()), "embed_fwd_shard")
        count_launches()
        if world > 1:
            out = torch.empty(Bsz, Ln, d, device=tok.device, dtype=torch.float32)
            dist.reduce_scatter_tensor(out, part, op=dist.ReduceOp.SUM, group=group)
        else:
            out = part
        ctx.save_for_backward(tok, tok_all)
        ctx.meta = (table_shard.shape, pos.shape, int(v_begin), v_end, float(scale), int(zero_pad), float(p), seed, site, group, world, rank,
                    float(grad_unscale))
        return out

    @staticmethod
    def backward(ctx, dout):
        from . import ops
        lib = L.load()
        tok, tok_all = ctx.saved_tensors
        tshape, pshape, v_begin, v_end, scale, zero_pad, p, seed, site, group, world, rank, unscale = ctx.meta
        Bsz, Ln = tok.shape
        d = tshape[1]
        dout = dout.contiguous()
        g = torch.empty_like(dout)
        dpos = torch.zeros(pshape, device=dout.device, dtype=torch.float32)
        check(lib.rbm_embed_bwd_offset(ptr(tok), ptr(dout), ptr(g), ptr(dpos), Bsz * Ln, Ln, d, zero_pad, p, seed, site, rank * Bsz * Ln,
                                       stream()), "embed_bwd_offset")
        count_launches()
        if world > 1:
            g_all = torch.empty(world * Bsz, Ln, d, device=dout.device, dtype=torch.float32)
            dist.all_gather_into_tensor(g_all, g, group=group)
        else:
            g_all = g
        keys = shard_keys(tok_all.reshape(-1), v_begin, v_end)
        rows = tshape[0]
        dtable = torch.zeros(rows, d, device=dout.device, dtype=torch.float32)
        ops.scatter_add_sorted_(dtable, keys, g_all.reshape(-1, d), None, scale / unscale, padding_idx=rows, vocab=rows + 1)
        return None, dtable, dpos, None, None, None, None, None, None, None, None, None


def sharded_embedding(tok, table_shard, pos, v_begin: int, vocab: int, scale: float, zero_pad: int, p: float, seed: int, site: int,
                      group=None, grad_unscale: float = 1.0):
    """See ShardedEmbedFn.  ``table_shard`` = rows ``shard_range(vocab, rank, world)`` of the [vocab, d] table."""
    return ShardedEmbedFn.apply(tok, table_shard, pos, v_begin, vocab, scale, zero_pad, p, seed, site, group, grad_unscale)


# ------------------------------------------------- BASELINE configs[3] layout: data-parallel body, row-sharded item tables
def shard_bert_model(model, group=None, capacity=None):
    """Cut ``bert.embedding.token.weight [V+2, d]``, ``out.weight [V+1, d]`` and ``out.bias`` of a BERT4Rec model down to this
    rank's row blocks (``shard_range``), in place; ``hidden_states`` / ``loss`` then go through :func:`sharded_embedding` and
    :func:`hybrid_vocab_parallel_loss`.  Build the model identically on every rank first (same ``model_init_seed``), shard, then
    create the optimizer; give ``GradSync`` only :func:`replicated_parameters`.  ``capacity`` = slots for labelled rows per rank in
    the loss exchange (None: all rows).  Dropout: the embedding site uses the common seed with global element indices, the body
    sites a rank-specific seed (independent masks per rank).  ``full_catalogue_topk`` of a sharded model goes through
    :func:`sharded_model_topk`, ``candidate_scores`` through :func:`sharded_candidate_scores`; ``forward`` (materialised logits)
    stays single-GPU only."""
    import types
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    tok = model.bert.embedding.token
    tok_rows, out_rows = tok.weight.shape[0], model.out.weight.shape[0]
    tb, te = shard_range(tok_rows, rank, world)
    ob, oe = shard_range(out_rows, rank, world)
    tok.weight = torch.nn.Parameter(tok.weight.data[tb:te].clone())
    model.out.weight = torch.nn.Parameter(model.out.weight.data[ob:oe].clone())
    model.out.bias = torch.nn.Parameter(model.out.bias.data[ob:oe].clone())
    for p in (tok.weight, model.out.weight, model.out.bias):
        p._rbm_sharded = True
    model._shard = types.SimpleNamespace(group=group, rank=rank, world=world, tok_begin=tb, tok_rows=tok_rows, out_begin=ob,
                                         out_rows=out_rows, capacity=capacity, overflow=None)
    return model


def replicated_parameters(model):
    """The parameters every rank holds whole (what ``GradSync`` averages); row-sharded tensors are updated locally."""
    return [p for p in model.parameters() if not getattr(p, "_rbm_sharded", False)]


def decorrelate_dropout(model, group=None):
    """Give each data-parallel rank its own dropout stream (ranks are built from the same seeds otherwise)."""
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    model.dropout_seed = (int(model.dropout_seed) + rank * 0x9E3779B97F4A7C15) & 0x7FFFFFFFFFFFFFFF
    return model


def _score_layer(model):
    """(weight shard, bias shard or None, first global row of the shard) of the layer the catalogue is scored against:
    BERT4Rec's untied ``out`` Linear (NN/models/bert.py:10), SASRec's item table itself (NN/models/sas_model/sas.py:110)."""
    sh = model._shard
    if hasattr(model, "out"):
        return model.out.weight, model.out.bias, sh.out_begin
    return model.sas.item_emb.weight, None, sh.tok_begin


def sharded_model_topk(model, x, k: int = 10, exclude=None):
    """Full-catalogue top-k of the last position for a model cut by :func:`shard_bert_model` / :func:`shard_sas_model`
    (SURVEY.md 8e, top-k eval): the last hidden rows of all ranks' users are all-gathered ([B, d] per rank), every rank runs
    the fused scoring + top-k on ITS rows of the scored layer with GLOBAL item ids, the per-shard lists are exchanged with an
    all-to-all by user range (each rank receives the lists of its own users only: k * 12 B per user and shard) and merged
    under the single-GPU order rule (score desc, id asc), so the result equals the unsharded model's.  Every rank must pass
    the same number of users.  ``exclude`` ([B, n] global item ids of this rank's users, see ``ops.score_topk``; every rank
    passes one or every rank passes None) travels with the hidden rows: padded to the largest n of all ranks and all-gathered,
    so every shard filters every user with global ids."""
    from . import ops
    sh = model._shard
    group, world, rank = sh.group, sh.world, sh.rank
    h = model.last_hidden(x).contiguous()
    B, d = h.shape
    if exclude is not None:
        exclude = model._device_long(exclude).reshape(B, -1)
    if world > 1:
        h_all = torch.empty(world * B, d, device=h.device, dtype=h.dtype)
        dist.all_gather_into_tensor(h_all, h, group=group)
        if exclude is not None:
            n = torch.tensor([exclude.shape[1]], device=h.device, dtype=torch.int64)
            dist.all_reduce(n, op=dist.ReduceOp.MAX, group=group)
            n = int(n.item())
            padded = torch.zeros(B, n, device=h.device, dtype=torch.int64)
            padded[:, :exclude.shape[1]] = exclude
            exclude = torch.empty(world * B, n, device=h.device, dtype=torch.int64)
            dist.all_gather_into_tensor(exclude, padded, group=group)
    else:
        h_all = h
    w, b, begin = _score_layer(model)
    lo = 1 if begin == 0 else 0  # row 0 is the padding id, not an item
    if w.shape[0] > lo:
        vals, ids = ops.score_topk(h_all, w, b, lo, w.shape[0], k, id_offset=begin, exclude=exclude)
    else:
        vals = torch.full((world * B, k), float("-inf"), device=h.device)
        ids = torch.full((world * B, k), -1, device=h.device, dtype=torch.int64)
    if world == 1:
        return vals, ids
    rv, ri = torch.empty_like(vals), torch.empty_like(ids)
    dist.all_to_all_single(rv, vals.contiguous(), group=group)  # chunk s of the result = shard s's lists for MY users
    dist.all_to_all_single(ri, ids.contiguous(), group=group)
    return ops.topk_merge(rv.view(world, B, k), ri.view(world, B, k))


# ------------------------------------------------------- sampled-candidate scoring / SASRec pos-neg scoring, sharded table
def owned_local_ids(ids: torch.Tensor, v_begin: int, v_end: int):
    """(local row index, owned mask) of global item ids against the row block [v_begin, v_end): rows of other blocks (and
    nothing else) are redirected to local row 0 with ``owned = False`` -- their contribution is multiplied by zero."""
    owned = (ids >= v_begin) & (ids < v_end)
    return torch.where(owned, ids - v_begin, torch.zeros_like(ids)), owned


def sharded_candidate_scores(model, x, candidates):
    """``scores[u, c] = <table[cand[u, c]], h_last[u]> (+ bias)`` (NN/models/sas_model/sas.py:110-114, NN/trainers/bert.py:47-49)
    for a row-sharded model: hidden rows and candidate ids of all ranks are all-gathered, every rank scores the candidates whose
    rows it holds (``rbm_candidate_scores``; the others count as exact zeros), and a reduce-scatter returns each rank the
    scores of its own users -- one non-zero addend per element, so the value equals the unsharded model's bit for bit."""
    from . import ops
    sh = model._shard
    group, world = sh.group, sh.world
    h = model.last_hidden(x).contiguous()
    cand = model._device_long(candidates)
    B, d = h.shape
    if world > 1:
        h_all = torch.empty(world * B, d, device=h.device, dtype=h.dtype)
        c_all = torch.empty(world * B, cand.shape[1], device=h.device, dtype=cand.dtype)
        dist.all_gather_into_tensor(h_all, h, group=group)
        dist.all_gather_into_tensor(c_all, cand, group=group)
    else:
        h_all, c_all = h, cand
    w, b, begin = _score_layer(model)
    loc, owned = owned_local_ids(c_all, begin, begin + w.shape[0])
    part = ops.candidate_scores(h_all, w, b, loc) * owned.to(torch.float32)
    if world == 1:
        return part
    out = torch.empty(B, cand.shape[1], device=h.device, dtype=torch.float32)
    dist.reduce_scatter_tensor(out, part.contiguous(), op=dist.ReduceOp.SUM, group=group)
    return out


class ShardedSasScoreFn(torch.autograd.Function):
    """``pos/neg logits = <f, table[pos]>, <f, table[neg]>`` (NN/models/sas_model/sas.py:93-100) with the item table row-sharded
    and the sequences data-parallel.  Forward: feature rows and both id arrays are all-gathered, each rank takes the dot
    products of the ids it owns (``rbm_sas_score_fwd`` on redirected local ids, masked), reduce-scatter back to the owners of
    the sequences.  Backward: the logit gradients are all-gathered; ``df`` shares (``rbm_sas_score_bwd`` with the gradients of
    ids the rank does not own set to zero) are reduce-scattered; the table-shard gradient is the deterministic
    sort/segment-reduce over the gathered rows with the not-owned positions keyed to the skipped row.  ``grad_unscale`` as in
    :class:`ShardedEmbedFn`."""

    @staticmethod
    def forward(ctx, f, table_shard, pos, neg, v_begin, group, grad_unscale):
        from . import ops
        lib = L.load()
        L.require_cuda(f, table_shard, pos, neg)
        world = dist.get_world_size(group) if dist.is_initialized() else 1
        f2 = f.reshape(-1, f.shape[-1]).contiguous()
        n, d = f2.shape
        pos, neg = pos.reshape(-1).contiguous(), neg.reshape(-1).contiguous()
        if world > 1:
            f_all = torch.empty(world * n, d, device=f.device, dtype=torch.float32)
            p_all, n_all = torch.empty(world * n, device=f.device, dtype=pos.dtype), torch.empty(world * n, device=f.device, dtype=neg.dtype)
            dist.all_gather_into_tensor(f_all, f2, group=group)
            dist.all_gather_into_tensor(p_all, pos, group=group)
            dist.all_gather_into_tensor(n_all, neg, group=group)
        else:
            f_all, p_all, n_all = f2, pos, neg
        v_end = int(v_begin) + table_shard.shape[0]
        pl_, po = owned_local_ids(p_all, int(v_begin), v_end)
        nl_, no = owned_local_ids(n_all, int(v_begin), v_end)
        pl = torch.empty(world * n, device=f.device, dtype=torch.float32)
        nl = torch.empty(world * n, device=f.device, dtype=torch.float32)
        check(lib.rbm_sas_score_fwd(ptr(f_all), ptr(table_shard), ptr(pl_), ptr(nl_), ptr(pl), ptr(nl), world * n, d, stream()), "sas_score_fwd")
        count_launches()
        both = torch.stack([pl * po.to(torch.float32), nl * no.to(torch.float32)], 1)  # [world*n, 2]
        if world > 1:
            mine = torch.empty(n, 2, device=f.device, dtype=torch.float32)
            dist.reduce_scatter_tensor(mine, both.contiguous(), op=dist.ReduceOp.SUM, group=group)
        else:
            mine = both
        ctx.save_for_backward(f_all, table_shard, p_all, n_all, pl_, nl_, po, no)
        ctx.meta = (f.shape, n, d, int(v_begin), v_end, group, world, float(grad_unscale))
        return mine[:, 0].reshape(f.shape[:-1]), mine[:, 1].reshape(f.shape[:-1])

    @staticmethod
    def backward(ctx, dpl, dnl):
        from . import ops
        lib = L.load()
        f_all, table_shard, p_all, n_all, pl_, nl_, po, no = ctx.saved_tensors
        fshape, n, d, v_begin, v_end, group, world, unscale = ctx.meta
        g = torch.stack([dpl.reshape(-1), dnl.reshape(-1)], 1).contiguous().float()
        if world > 1:
            g_all = torch.empty(world * n, 2, device=g.device, dtype=torch.float32)
            dist.all_gather_into_tensor(g_all, g, group=group)
        else:
            g_all = g
        dp = (g_all[:, 0] * po.to(torch.float32)).contiguous()
        dn = (g_all[:, 1] * no.to(torch.float32)).contiguous()
        df_all = torch.empty_like(f_all)
        check(lib.rbm_sas_score_bwd(ptr(table_shard), ptr(pl_), ptr(nl_), ptr(dp), ptr(dn), ptr(df_all), world * n, d, stream()), "sas_score_bwd")
        count_launches()
        if world > 1:
            df = torch.empty(n, d, device=g.device, dtype=torch.float32)
            dist.reduce_scatter_tensor(df, df_all, op=dist.ReduceOp.SUM, group=group)
        else:
            df = df_all
        rows = table_shard.shape[0]
        dtable = torch.zeros(rows, d, device=g.device, dtype=torch.float32)
        ops.scatter_add_sorted_(dtable, shard_keys(p_all, v_begin, v_end), f_all, dp, 1.0 / unscale, padding_idx=rows, vocab=rows + 1)
        ops.scatter_add_sorted_(dtable, shard_keys(n_all, v_begin, v_end), f_all, dn, 1.0 / unscale, padding_idx=rows, vocab=rows + 1)
        return df.view(fshape), dtable, None, None, None, None, None


def shard_sas_model(model, group=None):
    """Cut ``sas.item_emb.weight [V+1, d]`` of a SASRec model down to this rank's row block, in place (SURVEY.md 8e): the input
    lookup goes through :func:`sharded_embedding`, the pos/neg scoring through :class:`ShardedSasScoreFn`, ``predict`` through
    :func:`sharded_candidate_scores` and ``full_catalogue_topk`` through :func:`sharded_model_topk`; sequences stay
    data-parallel, ``GradSync(replicated_parameters(model))`` averages the dense body.  Build the model identically on every
    rank first (same torch seed), shard, then create the optimizer."""
    import types
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    emb = model.sas.item_emb
    rows = emb.weight.shape[0]
    b, e = shard_range(rows, rank, world)
    emb.weight = torch.nn.Parameter(emb.weight.data[b:e].clone())
    emb.weight._rbm_sharded = True
    model._shard = types.SimpleNamespace(group=group, rank=rank, world=world, tok_begin=b, tok_rows=rows, capacity=None, overflow=None)
    return model
