"""BERT4Rec with the reference's constructor, ``forward`` and ``state_dict`` (NN/models/bert.py:6-16,
NN/models/bert_modules/**), computed by the sm_100a kernels of librbm_b200.

The nn.Module tree below only *holds parameters* under the reference's names -- so checkpoints interchange and, being
built from the same torch layers in the same order after ``fix_random_seed_as(model_init_seed)``
(NN/models/bert_modules/bert.py:12), the initial weights are bit-identical to the reference's.  None of these holder
modules' own ``forward`` is ever used.
"""
import math
import os
import random

import numpy as np
import torch
import torch.nn as nn

from .. import lib as L
from .. import ops
from .base import BaseModel


def fix_random_seed_as(random_seed):
    """NN/utils.py:65-71."""
    random.seed(random_seed)
    torch.manual_seed(random_seed)
    torch.cuda.manual_seed_all(random_seed)
    np.random.seed(random_seed)
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False


class _Norm(nn.Module):  # NN/models/bert_modules/utils/layer_norm.py:8-12 (a_2, b_2, eps=1e-6)
    def __init__(self, size):
        super().__init__()
        self.a_2 = nn.Parameter(torch.ones(size))
        self.b_2 = nn.Parameter(torch.zeros(size))
        self.eps = 1e-6


class _Sublayer(nn.Module):  # NN/models/bert_modules/utils/sublayer.py:11-14
    def __init__(self, size):
        super().__init__()
        self.norm = _Norm(size)


class _Attention(nn.Module):  # NN/models/bert_modules/attention/multi_head.py:10-22
    def __init__(self, h, d_model):
        super().__init__()
        assert d_model % h == 0
        self.d_k = d_model // h
        self.h = h
        self.linear_layers = nn.ModuleList([nn.Linear(d_model, d_model) for _ in range(3)])
        self.output_linear = nn.Linear(d_model, d_model)


class _FeedForward(nn.Module):  # NN/models/bert_modules/utils/feed_forward.py:8-13
    def __init__(self, d_model, d_ff):
        super().__init__()
        self.w_1 = nn.Linear(d_model, d_ff)
        self.w_2 = nn.Linear(d_ff, d_model)


class _Block(nn.Module):  # NN/models/bert_modules/transformer.py:13-26
    def __init__(self, hidden, heads, ff_hidden):
        super().__init__()
        self.attention = _Attention(heads, hidden)
        self.feed_forward = _FeedForward(hidden, ff_hidden)
        self.input_sublayer = _Sublayer(hidden)
        self.output_sublayer = _Sublayer(hidden)


class _Token(nn.Embedding):  # NN/models/bert_modules/embedding/token.py:4-6
    def __init__(self, vocab_size, embed_size):
        super().__init__(vocab_size, embed_size, padding_idx=0)


class _Position(nn.Module):  # NN/models/bert_modules/embedding/position.py:8-12
    def __init__(self, max_len, d_model):
        super().__init__()
        self.pe = nn.Embedding(max_len, d_model)


class _Embedding(nn.Module):  # NN/models/bert_modules/embedding/bert.py:17-27
    def __init__(self, vocab_size, embed_size, max_len):
        super().__init__()
        self.token = _Token(vocab_size, embed_size)
        self.position = _Position(max_len, embed_size)


class BERT(nn.Module):
    """Parameter tree of NN/models/bert_modules/bert.py:8-34."""

    def __init__(self, args):
        super().__init__()
        fix_random_seed_as(args.model_init_seed)
        self.max_len = args.max_len
        self.hidden = args.bert_hidden_units
        self.heads = args.bert_num_heads
        self.n_layers = args.bert_num_blocks
        self.p_attn = float(args.bert_dropout)
        self.p_hidden = float(args.bert_hidden_dropout)
        vocab_size = args.num_items + 2  # [MASK] = num_items + 1, padding = 0
        self.embedding = _Embedding(vocab_size, self.hidden, self.max_len)
        self.transformer_blocks = nn.ModuleList([_Block(self.hidden, self.heads, self.hidden * 4) for _ in range(self.n_layers)])


class BERTModel(BaseModel):
    def __init__(self, args):
        super().__init__(args)
        self.bert = BERT(args)
        self.out = nn.Linear(self.bert.hidden, args.num_items + 1)
        self.num_items = args.num_items

    @classmethod
    def code(cls):
        return 'bert'

    # ------------------------------------------------------------------ transformer body (a7-a11)
    def hidden_states(self, x, last_only=False, label_rows=None):
        """BERT.forward NN/models/bert_modules/bert.py:36-43 -> [B, L, d]; ``last_only`` (evaluation, K20): [B, d], the last position
        alone, with the final block computed for that position only (keys / values still from every position).  ``label_rows``
        (training, an ``ops.LiveRows`` over the labels): [cap, d], the labelled positions alone -- the loss reads no other row of the
        final block's output, so its output projection, LayerNorm and feed-forward run on those rows only."""
        bert = self.bert
        tok = self._device_long(x)
        Bsz, Ln = tok.shape
        if Ln != bert.max_len:
            raise RuntimeError("BERT4Rec adds the whole positional table: sequence length %d must equal max_len %d "
                               "(NN/models/bert_modules/embedding/position.py:16)" % (Ln, bert.max_len))
        d, h = bert.hidden, bert.heads
        train = self.training
        p_h = bert.p_hidden if train else 0.0
        p_a = bert.p_attn if train else 0.0
        seed = self.dropout_seed
        base = self._next_site_base() if train else 0
        sh = getattr(self, "_shard", None)
        if sh is None:
            x = ops.EmbedFn.apply(tok, bert.embedding.token.weight, bert.embedding.position.pe.weight, 1.0, 0, p_h, seed, base)
        else:  # row-sharded item table (rbm_b200.dist.shard_bert_model): common seed + global element indices for this site,
            #    a rank-specific seed for the body sites
            from ..dist import sharded_embedding
            x = sharded_embedding(tok, bert.embedding.token.weight, bert.embedding.position.pe.weight, sh.tok_begin, sh.tok_rows, 1.0, 0,
                                  p_h, seed, base, sh.group, grad_unscale=float(sh.world))
            seed = (seed + (sh.rank + 1) * 0x9E3779B97F4A7C15) & 0x7FFFFFFFFFFFFFFF
        scale = 1.0 / math.sqrt(d // h)
        for b, blk in enumerate(bert.transformer_blocks):
            s = base + 1 + 5 * b
            att, ff = blk.attention, blk.feed_forward
            if last_only and b == len(bert.transformer_blocks) - 1:
                n1 = ops.layernorm(x, blk.input_sublayer.norm.a_2, blk.input_sublayer.norm.b_2, 1e-6, L.LN_BERT)
                lq, lk, lv = att.linear_layers
                kv = ops.linear(n1, torch.cat([lk.weight, lv.weight], 0), torch.cat([lk.bias, lv.bias], 0))
                ctx = ops.attention_last_query(ops.linear(n1[:, -1, :], lq.weight, lq.bias), kv, tok, Bsz, Ln, h, 0, d, L.MASK_KEYPAD, scale)
                xl = ops.linear(ctx, att.output_linear.weight, att.output_linear.bias, residual=x[:, -1, :])
                n2 = ops.layernorm(xl, blk.output_sublayer.norm.a_2, blk.output_sublayer.norm.b_2, 1e-6, L.LN_BERT)
                u = ops.linear(n2, ff.w_1.weight, ff.w_1.bias, act=L.ACT_GELU_TANH)
                return ops.linear(u, ff.w_2.weight, ff.w_2.bias, residual=xl)
            lq = getattr(label_rows, "lq", None) if (label_rows is not None and b == len(bert.transformer_blocks) - 1) else None
            lq_path = lq is not None and ops.attention_lq_supported(Ln, lq, d // h, L.MASK_KEYPAD)
            if lq_path:  # the normalised rows feed two consumers here (k / v of every row, q of the labelled rows): their gradients
                #          and the residual one meet inside the LayerNorm-backward launch
                n1, n1q, x = ops.layernorm_fanout(x, blk.input_sublayer.norm.a_2, blk.input_sublayer.norm.b_2, 1e-6, L.LN_BERT)
            else:
                n1, x = ops.layernorm_residual(x, blk.input_sublayer.norm.a_2, blk.input_sublayer.norm.b_2, 1e-6, L.LN_BERT)
            if lq_path:
                # final block, labelled rows: queries of those rows only (<= lq per sequence, compacted per sequence) against the
                # keys / values of every position; the attention site indexes its Philox stream by (sequence-head, query ordinal, key)
                wq, wk, wv = att.linear_layers
                kv = ops.linear(n1, torch.cat([wk.weight, wv.weight], 0), torch.cat([wk.bias, wv.bias], 0))
                qc = ops.linear(ops.rows_gather(n1q.view(-1, d), label_rows), wq.weight, wq.bias)
                ctx = ops.attention_lq(ops.rows_to_seq(qc, label_rows, Bsz, Ln, lq), kv, tok, Bsz, Ln, lq, h, L.MASK_KEYPAD, scale, p_a,
                                       seed, s)
                ctx = ops.seq_to_rows(ctx, label_rows, Bsz, Ln, lq)
                xc = ops.linear(ctx, att.output_linear.weight, att.output_linear.bias, residual=ops.rows_gather(x.view(-1, d), label_rows),
                                pA=p_h, siteA=s + 1, seed=seed)
                n2, xc = ops.layernorm_residual(xc, blk.output_sublayer.norm.a_2, blk.output_sublayer.norm.b_2, 1e-6, L.LN_BERT)
                u = ops.linear(n2, ff.w_1.weight, ff.w_1.bias, act=L.ACT_GELU_TANH, pA=p_h, siteA=s + 2, seed=seed)
                return ops.linear(u, ff.w_2.weight, ff.w_2.bias, residual=xc, pA=p_h, siteA=s + 3, pB=p_h, siteB=s + 4, seed=seed)
            w_qkv = torch.cat([l.weight for l in att.linear_layers], 0)
            b_qkv = torch.cat([l.bias for l in att.linear_layers], 0)
            qkv = ops.linear(n1, w_qkv, b_qkv)
            ctx = ops.attention(qkv, None, tok, Bsz, Ln, h, 0, d, 2 * d, L.MASK_KEYPAD, scale, p_a, seed, s)
            if label_rows is not None and b == len(bert.transformer_blocks) - 1:
                # the rest of the final block on the labelled rows only (their element-wise dropout sites index the Philox stream
                # by (labelled-row ordinal, column)); keys / values above came from every position
                xc = ops.linear(ops.rows_gather(ctx.view(-1, d), label_rows), att.output_linear.weight, att.output_linear.bias,
                                residual=ops.rows_gather(x.view(-1, d), label_rows), pA=p_h, siteA=s + 1, seed=seed)
                n2, xc = ops.layernorm_residual(xc, blk.output_sublayer.norm.a_2, blk.output_sublayer.norm.b_2, 1e-6, L.LN_BERT)
                u = ops.linear(n2, ff.w_1.weight, ff.w_1.bias, act=L.ACT_GELU_TANH, pA=p_h, siteA=s + 2, seed=seed)
                return ops.linear(u, ff.w_2.weight, ff.w_2.bias, residual=xc, pA=p_h, siteA=s + 3, pB=p_h, siteB=s + 4, seed=seed)
            x = ops.linear(ctx.view(Bsz, Ln, d), att.output_linear.weight, att.output_linear.bias, residual=x, pA=p_h,
                           siteA=s + 1, seed=seed)
            n2, x = ops.layernorm_residual(x, blk.output_sublayer.norm.a_2, blk.output_sublayer.norm.b_2, 1e-6, L.LN_BERT)
            u = ops.linear(n2, ff.w_1.weight, ff.w_1.bias, act=L.ACT_GELU_TANH, pA=p_h, siteA=s + 2, seed=seed)
            x = ops.linear(u, ff.w_2.weight, ff.w_2.bias, residual=x, pA=p_h, siteA=s + 3, pB=p_h, siteB=s + 4, seed=seed)
        return x

    # ------------------------------------------------------------------ reference API
    def forward(self, x):
        """NN/models/bert.py:15-16: logits [B, L, V+1].  Compatibility path that materialises the logits (small shapes,
        parity tests); training uses :meth:`loss`, evaluation :meth:`candidate_scores` / :meth:`full_catalogue_topk`."""
        self._unsharded_only("forward")
        h = self.hidden_states(x)
        V1 = self.out.weight.shape[0]
        pad = (-V1) % 4
        w, b = self.out.weight, self.out.bias
        if pad:
            w = torch.cat([w, w.new_zeros(pad, w.shape[1])], 0)
            b = torch.cat([b, b.new_zeros(pad)], 0)
        logits = ops.linear(h, w, b)
        return logits[..., :V1].contiguous() if pad else logits

    # ------------------------------------------------------------------ fused paths used by the drop-in trainer
    def loss(self, x, labels):
        """CE(ignore_index=0) of NN/trainers/bert.py:30-41 without materialising [B*L, V+1] logits (K15-K16)."""
        sh = getattr(self, "_shard", None)
        if sh is None and self.training:
            lab = self._device_long(labels)
            live = self._label_rows(lab)
            if live is not None:  # final block and scoring on the labelled rows only
                return ops.score_cross_entropy(self.hidden_states(x, label_rows=live), live.ids, self.out.weight, self.out.bias)
        h = self.hidden_states(x)
        if sh is not None:  # data-parallel rows x row-sharded output layer: the loss of the GLOBAL batch (SURVEY 8e)
            from ..dist import hybrid_vocab_parallel_loss
            loss, sh.overflow = hybrid_vocab_parallel_loss(h, self._device_long(labels), self.out.weight, self.out.bias, sh.out_begin,
                                                           sh.capacity, sh.group)
            # accumulated on the device; the trainer asserts it once per epoch (trainers/base.py _check_shard_overflow)
            sh.overflow_any = sh.overflow if getattr(sh, "overflow_any", None) is None else (sh.overflow_any | sh.overflow)
            return loss
        return ops.score_cross_entropy(h, self._device_long(labels), self.out.weight, self.out.bias)

    # ------------------------------------------------------------------ labelled-row path (training)
    LABEL_ROWS_MAX_FRACTION = 0.5  # above this share of labelled positions the final block runs on every row

    def _label_rows(self, labels):
        """``ops.LiveRows`` over the labelled positions (``.lq``: an upper bound on the labelled positions of one sequence, None =
        keep every query in the final block's attention), or None (final block on every row).  Eager steps read the counts back
        (one host sync); under a CUDA graph the trainer fixes both capacities before capture (``_row_cap``: rows, 0 = off;
        ``_graph_lq``) and checks every replayed batch against them."""
        if os.environ.get("RBM_BERT_LABEL_ROWS", "1") == "0":
            return None
        n, Ln = labels.numel(), labels.shape[-1]
        cap = getattr(self, "_row_cap", None)
        if cap is None:
            cnt, mx = self._label_counts(labels)
            if cnt > self.LABEL_ROWS_MAX_FRACTION * n:
                return None
            cap, lq = self._capacities(cnt, mx)  # the same rule a captured step is sized by
        elif cap <= 0:
            return None
        else:
            lq = getattr(self, "_graph_lq", None)
        live = ops.LiveRows(labels, cap, keep_ids=True)
        live.lq = lq if (lq is not None and lq < Ln and os.environ.get("RBM_BERT_LABEL_QUERIES", "1") != "0") else None
        return live

    @staticmethod
    def _capacities(cnt: int, mx: int):
        """(row capacity, per-sequence query capacity) for a batch with ``cnt`` labelled positions, at most ``mx`` in one sequence:
        headroom 12.5 % + 8 sqrt(cnt) rows (a batch's count is a sum over its sequences: small batches vary more) resp. 25 % + 8,
        rounded to the kernels' tiles.  Eager steps and captured steps use the same rule, so a step replayed from a
        graph captured on a batch with the same counts is bit-identical to the eager step."""
        return -(-(cnt + cnt // 8 + 8 * math.isqrt(cnt) + 64) // 128) * 128, -(-(mx + mx // 4 + 8) // 16) * 16

    @staticmethod
    def _label_counts(labels):
        """(labelled positions of the batch, most labelled positions of one sequence) -- one device -> host read."""
        labels = torch.as_tensor(labels)
        per = torch.count_nonzero(labels.reshape(-1, labels.shape[-1]), dim=1)
        cnt, mx = torch.stack([per.sum(), per.max()]).tolist()
        return int(cnt), int(mx)

    def row_capacity_for(self, tokens, labels) -> int:
        """Capacity (rows) a captured step should be built with for batches like this one: headroom over its labelled rows (``_capacities``)
        (0 = run the final block on every row), and the per-sequence query capacity ``_graph_lq`` of the final block's attention.
        ``live_row_count`` tells the trainer whether a later batch still fits."""
        self._graph_lq = None
        if os.environ.get("RBM_BERT_LABEL_ROWS", "1") == "0" or getattr(self, "_shard", None) is not None:
            return 0
        labels = torch.as_tensor(labels)
        n, Ln = int(labels.numel()), int(labels.shape[-1])
        cnt, mx = self._label_counts(labels)
        if cnt > self.LABEL_ROWS_MAX_FRACTION * n:
            return 0
        cap, lq = self._capacities(cnt, mx)
        self._graph_lq = lq if lq < Ln else None
        return min(cap, -(-n // 128) * 128)

    def live_row_count(self, tokens, labels) -> int:
        """Labelled rows of the batch -- or more than any capacity when one sequence has more labels than the captured step's
        per-sequence query capacity."""
        cnt, mx = self._label_counts(labels)
        lq = getattr(self, "_graph_lq", None)
        return (1 << 60) if (lq is not None and mx > lq) else cnt

    def last_hidden(self, x):
        if not self.training and not torch.is_grad_enabled():
            return self.hidden_states(x, last_only=True)
        return self.hidden_states(x)[:, -1, :]

    def _unsharded_only(self, what):
        if getattr(self, "_shard", None) is not None:
            raise RuntimeError("%s: not wired for a row-sharded model (use full_catalogue_topk, or gather the tables with "
                               "rbm_b200.checkpoint)" % what)

    def candidate_scores(self, x, candidates):
        """scores[:, -1, :].gather(1, candidates) of NN/trainers/bert.py:47-49, scoring only the candidates."""
        if getattr(self, "_shard", None) is not None:
            from ..dist import sharded_candidate_scores
            return sharded_candidate_scores(self, x, candidates)
        return ops.candidate_scores(self.last_hidden(x), self.out.weight, self.out.bias, self._device_long(candidates))

    def full_catalogue_topk(self, x, k=10, exclude=None):
        """Top-k items (ids 1..V) of the last position, (score desc, id asc); scores never materialised (K19-K21).
        ``exclude`` ([B, n] int64 item ids, ids <= 0 = padding): items each user must not be ranked, e.g. their history."""
        if getattr(self, "_shard", None) is not None:
            from ..dist import sharded_model_topk
            return sharded_model_topk(self, x, k, exclude=exclude)
        return ops.score_topk(self.last_hidden(x), self.out.weight, self.out.bias, 1, self.num_items + 1, k,
                              exclude=self._device_long(exclude) if exclude is not None else None)
