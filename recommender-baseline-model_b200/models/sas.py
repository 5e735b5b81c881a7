"""SASRec with the reference's constructor, ``forward`` / ``predict`` and ``state_dict`` (NN/models/sas.py:6-19,
NN/models/sas_model/sas.py:24-118), computed by the sm_100a kernels of librbm_b200.

``self.sas`` holds parameters under the reference's names, built from the same torch layers in the same order (so a
given torch seed yields the reference's initial weights); their own ``forward`` is never used.
"""
import math
import os

import torch
import torch.nn as nn

from .. import lib as L
from .. import ops
from .base import BaseModel


class _PointWiseFeedForward(nn.Module):  # NN/models/sas_model/sas.py:7-14
    def __init__(self, hidden_units):
        super().__init__()
        self.conv1 = nn.Conv1d(hidden_units, hidden_units, kernel_size=1)
        self.conv2 = nn.Conv1d(hidden_units, hidden_units, kernel_size=1)


class SAS(nn.Module):
    """Parameter tree of NN/models/sas_model/sas.py:24-57."""

    def __init__(self, args):
        super().__init__()
        self.item_num = args.num_items
        d = args.sas_hidden_units
        self.hidden = d
        self.heads = args.sas_heads
        self.p = float(args.sas_dropout)
        self.item_emb = nn.Embedding(self.item_num + 1, d, padding_idx=0)
        self.pos_emb = nn.Embedding(args.max_len, d)
        self.attention_layernorms = nn.ModuleList()
        self.attention_layers = nn.ModuleList()
        self.forward_layernorms = nn.ModuleList()
        self.forward_layers = nn.ModuleList()
        self.last_layernorm = nn.LayerNorm(d, eps=1e-8)
        for _ in range(args.sas_num_blocks):
            self.attention_layernorms.append(nn.LayerNorm(d, eps=1e-8))
            self.attention_layers.append(nn.MultiheadAttention(d, self.heads, self.p))
            self.forward_layernorms.append(nn.LayerNorm(d, eps=1e-8))
            self.forward_layers.append(_PointWiseFeedForward(d))


class SASModel(BaseModel):
    def __init__(self, args):
        super().__init__(args)
        self.sas = SAS(args)

    @classmethod
    def code(cls):
        return 'sas'

    def log2feats(self, log_seqs, last_only=False, live=None):
        """SAS.log2feats NN/models/sas_model/sas.py:59-88 -> [B, L, d]; ``last_only`` (evaluation, K20): [B, d], the last position's
        features, with the final block computed for that position alone (keys / values still from every position)."""
        sas = self.sas
        seq = self._device_long(log_seqs)
        Bsz, Ln = seq.shape
        d, h = sas.hidden, sas.heads
        train = self.training
        p = sas.p if train else 0.0
        seed = self.dropout_seed
        base = self._next_site_base() if train else 0
        sh = getattr(self, "_shard", None)
        if live is None and sh is None and (train or (last_only and not torch.is_grad_enabled())):
            live = self._live_rows(seq)  # training, and evaluation of the last position: token-wise layers on the non-padding rows only
        if live is not None and live is not False:  # (False: the caller already decided for the dense path)
            return self._blocks_live_rows(seq, live, Bsz, Ln, p, seed, base, math.sqrt(1.0 / (d // h)), last_only)
        if sh is None:
            x = ops.EmbedFn.apply(seq, sas.item_emb.weight, sas.pos_emb.weight, float(d ** 0.5), 1, p, seed, base)
        else:  # row-sharded item table (rbm_b200.dist.shard_sas_model): common seed + global element indices for this site,
            #    a rank-specific seed for the body sites
            from ..dist import sharded_embedding
            x = sharded_embedding(seq, sas.item_emb.weight, sas.pos_emb.weight, sh.tok_begin, sh.tok_rows, float(d ** 0.5), 1, p, seed,
                                  base, sh.group, grad_unscale=float(sh.world))
            seed = (seed + (sh.rank + 1) * 0x9E3779B97F4A7C15) & 0x7FFFFFFFFFFFFFFF
        scale = math.sqrt(1.0 / (d // h))
        for b in range(len(sas.attention_layers)):
            s = base + 1 + 3 * b
            ln1, mha, ln2, ffn = sas.attention_layernorms[b], sas.attention_layers[b], sas.forward_layernorms[b], sas.forward_layers[b]
            # Q and x both have two consumers: layernorm_fanout hands out (Q, Q, x) so that the three gradients meet inside
            # the LayerNorm-backward launch instead of autograd's elementwise adds
            w_in, b_in = mha.in_proj_weight, mha.in_proj_bias
            if last_only and b == len(sas.attention_layers) - 1:
                Ql = ops.layernorm(x[:, -1, :], ln1.weight, ln1.bias, 1e-8, L.LN_TORCH)
                kv = ops.linear(x, w_in[d:], b_in[d:])
                ctx = ops.attention_last_query(ops.linear(Ql, w_in[:d], b_in[:d]), kv, None, Bsz, Ln, h, 0, d, L.MASK_CAUSAL, scale)
                xl = ops.linear(ctx, mha.out_proj.weight, mha.out_proj.bias, residual=Ql)
                xl = ops.layernorm(xl, ln2.weight, ln2.bias, 1e-8, L.LN_TORCH)
                u = ops.linear(xl, ffn.conv1.weight.squeeze(-1), ffn.conv1.bias, act=L.ACT_RELU)
                xl = ops.linear(u, ffn.conv2.weight.squeeze(-1), ffn.conv2.bias, residual=xl, row_tok=seq[:, -1])
                return ops.layernorm(xl, sas.last_layernorm.weight, sas.last_layernorm.bias, 1e-8, L.LN_TORCH)
            Q, Qres, xkv = ops.layernorm_fanout(x, ln1.weight, ln1.bias, 1e-8, L.LN_TORCH)
            q = ops.linear(Q, w_in[:d], b_in[:d])          # q from the normalised stream
            kv = ops.linear(xkv, w_in[d:], b_in[d:])       # k, v from the un-normalised stream (sas.py:75)
            ctx = ops.attention(q, kv, None, Bsz, Ln, h, 0, 0, d, L.MASK_CAUSAL, scale, p, seed, s)
            x = ops.linear(ctx.view(Bsz, Ln, d), mha.out_proj.weight, mha.out_proj.bias, residual=Qres)  # Q + mha (sas.py:79)
            x, xres, _ = ops.layernorm_fanout(x, ln2.weight, ln2.bias, 1e-8, L.LN_TORCH)
            u = ops.linear(x, ffn.conv1.weight.squeeze(-1), ffn.conv1.bias, act=L.ACT_RELU, pA=p, siteA=s + 1, seed=seed)
            x = ops.linear(u, ffn.conv2.weight.squeeze(-1), ffn.conv2.bias, residual=xres, row_tok=seq, pA=p, siteA=s + 2, seed=seed)
        return ops.layernorm(x, sas.last_layernorm.weight, sas.last_layernorm.bias, 1e-8, L.LN_TORCH)

    # ------------------------------------------------------------------ live-row path (training)
    LIVE_ROWS_MAX_FRACTION = 0.6  # above this share of non-padding rows the dense path is used

    def _live_rows(self, seq, *also):
        """Plan of the live-row path for this batch, or None for the dense path.  Eager steps read the number of non-padding
        positions back (one host sync); under a CUDA graph the trainer fixes the capacity before capture (``_row_cap``: rows,
        0 = dense) and checks every replayed batch against it.  ``also``: further id tensors (pos, neg) whose non-zero counts the
        capacity must cover too (their table-gradient scatters then run on ``cap`` entries)."""
        if os.environ.get("RBM_SAS_LIVE_ROWS", "1") == "0":
            return None
        n = seq.numel()
        cap = getattr(self, "_row_cap", None)
        if cap is None:
            cnts = torch.stack([torch.count_nonzero(t) for t in (seq,) + also]).tolist()
            if cnts[0] > self.LIVE_ROWS_MAX_FRACTION * n:
                return None
            cap = self._capacity(max(cnts))  # the same rule a captured step is sized by
        elif cap <= 0:
            return None
        live = ops.LiveRows(seq, cap)
        live.covers_labels = len(also) > 0
        return live

    def row_capacity_for(self, seq, *also) -> int:
        """Capacity (rows) a captured step should be built with for batches like (seq, pos, neg): headroom (``_capacity``) over the non-zero
        ids, 0 when the dense path is the better choice.  ``live_row_count`` tells the trainer whether a later batch still fits."""
        if os.environ.get("RBM_SAS_LIVE_ROWS", "1") == "0" or getattr(self, "_shard", None) is not None:
            return 0
        n, cnt = int(torch.as_tensor(seq).numel()), self.live_row_count(seq, *also)
        if int(torch.count_nonzero(torch.as_tensor(seq))) > self.LIVE_ROWS_MAX_FRACTION * n:
            return 0
        return min(self._capacity(cnt), -(-n // 128) * 128)

    @staticmethod
    def _capacity(cnt: int) -> int:
        """Row capacity for ``cnt`` non-zero ids: 12.5 % + 8 sqrt(cnt) rows of headroom (a batch's count is a sum over its sequences:
        small batches vary more), rounded to 128-row tiles (eager and captured steps alike)."""
        return -(-(cnt + cnt // 8 + 8 * math.isqrt(cnt) + 64) // 128) * 128

    @staticmethod
    def live_row_count(*ids) -> int:
        """The largest number of non-zero ids among the given tensors (seq, pos, neg of a batch)."""
        ts = [torch.as_tensor(t) for t in ids]
        return int(torch.stack([torch.count_nonzero(t) for t in ts]).max().item())

    def _blocks_live_rows(self, seq, live, Bsz, Ln, p, seed, base, scale, last_only=False):
        """The block loop with LayerNorm / Linear / feed-forward on the live rows only (csrc/rows.cu explains why that is exact).
        Attention runs on the same compact layout (csrc/attention_live.cu: every padding key of a sequence is the projection bias,
        which is what W.0 + b gives the reference, so they enter as one key with a multiplicity); sequences longer than 64 keep the
        dense kernels on the [B, L] layout (queries / keys / values scattered back).  The element-wise dropout sites of this path
        index their Philox stream by (live-row ordinal, column); the attention site by (sequence-head, i, j) as always.
        ``last_only`` (evaluation): [B, d], the final block for the last position alone, its keys / values from the compact rows."""
        sas = self.sas
        d, h = sas.hidden, sas.heads
        if ops.embed_live_supported(Ln, d):
            xc = ops.EmbedLiveFn.apply(seq, sas.item_emb.weight, sas.pos_emb.weight, live, float(d ** 0.5), p, seed, base)
        else:
            xc = ops.rows_gather(ops.EmbedFn.apply(seq, sas.item_emb.weight, sas.pos_emb.weight, float(d ** 0.5), 1, p, seed, base).view(-1, d), live)
        for b in range(len(sas.attention_layers)):
            s = base + 1 + 3 * b
            ln1, mha, ln2, ffn = sas.attention_layernorms[b], sas.attention_layers[b], sas.forward_layernorms[b], sas.forward_layers[b]
            w_in, b_in = mha.in_proj_weight, mha.in_proj_bias
            if last_only and b == len(sas.attention_layers) - 1:
                kv = ops.rows_scatter(ops.linear(xc, w_in[d:], b_in[d:]), b_in[d:], live)  # [B*L, 2d]; padding rows: the bias
                x_last = ops.rows_scatter(xc, None, live).view(Bsz, Ln, d)[:, -1, :]        # (a padding row is zero, as in the dense path)
                Ql = ops.layernorm(x_last, ln1.weight, ln1.bias, 1e-8, L.LN_TORCH)
                ctx = ops.attention_last_query(ops.linear(Ql, w_in[:d], b_in[:d]), kv, None, Bsz, Ln, h, 0, d, L.MASK_CAUSAL, scale)
                xl = ops.linear(ctx, mha.out_proj.weight, mha.out_proj.bias, residual=Ql)
                xl = ops.layernorm(xl, ln2.weight, ln2.bias, 1e-8, L.LN_TORCH)
                u = ops.linear(xl, ffn.conv1.weight.squeeze(-1), ffn.conv1.bias, act=L.ACT_RELU)
                xl = ops.linear(u, ffn.conv2.weight.squeeze(-1), ffn.conv2.bias, residual=xl, row_tok=seq[:, -1])
                return ops.layernorm(xl, sas.last_layernorm.weight, sas.last_layernorm.bias, 1e-8, L.LN_TORCH)
            Q, Qres, xkv = ops.layernorm_fanout(xc, ln1.weight, ln1.bias, 1e-8, L.LN_TORCH)
            q = ops.linear(Q, w_in[:d], b_in[:d])
            kv = ops.linear(xkv, w_in[d:], b_in[d:])
            if Ln <= 64 and d % h == 0 and d // h in (16, 32, 64, 128):  # compact attention: the padding keys of a sequence are one key with a multiplicity
                ctx = ops.attention_live(q, kv, b_in[d:], live, Bsz, Ln, h, scale, p, seed, s)
            else:  # dense attention kernels on the [B, L] layout (padding rows: zero queries, the bias as key / value)
                ctx = ops.attention(ops.rows_scatter(q, None, live), ops.rows_scatter(kv, b_in[d:], live), None, Bsz, Ln, h, 0, 0, d,
                                    L.MASK_CAUSAL, scale, p, seed, s)
                ctx = ops.rows_gather(ctx.view(-1, d), live)
            xc = ops.linear(ctx, mha.out_proj.weight, mha.out_proj.bias, residual=Qres)
            xc, xres, _ = ops.layernorm_fanout(xc, ln2.weight, ln2.bias, 1e-8, L.LN_TORCH)
            u = ops.linear(xc, ffn.conv1.weight.squeeze(-1), ffn.conv1.bias, act=L.ACT_RELU, pA=p, siteA=s + 1, seed=seed)
            xc = ops.linear(u, ffn.conv2.weight.squeeze(-1), ffn.conv2.bias, residual=xres, pA=p, siteA=s + 2, seed=seed)
        out = ops.layernorm(xc, sas.last_layernorm.weight, sas.last_layernorm.bias, 1e-8, L.LN_TORCH)
        return ops.rows_scatter(out, sas.last_layernorm.bias, live).view(Bsz, Ln, d)

    def forward(self, log_seqs, pos_seqs, neg_seqs):  # for training
        """NN/models/sas_model/sas.py:90-105 -> (pos_logits, neg_logits) [B, L]."""
        sh = getattr(self, "_shard", None)
        if sh is not None:
            from ..dist import ShardedSasScoreFn
            f = self.log2feats(log_seqs)
            return ShardedSasScoreFn.apply(f, self.sas.item_emb.weight, self._device_long(pos_seqs), self._device_long(neg_seqs),
                                           sh.tok_begin, sh.group, float(sh.world))
        pos, neg = self._device_long(pos_seqs), self._device_long(neg_seqs)
        live = (self._live_rows(self._device_long(log_seqs), pos, neg) or False) if self.training else None
        f = self.log2feats(log_seqs, live=live)
        return ops.sas_scores(f, self.sas.item_emb.weight, pos, neg, cap=live.cap if live else None)

    def loss(self, log_seqs, pos_seqs, neg_seqs):
        """BCE part of SASTrainer.calculate_loss NN/trainers/sas.py:34-49."""
        pos = self._device_long(pos_seqs)
        pl, nl = self.forward(log_seqs, pos, neg_seqs)
        loss = ops.bce_pair_loss(pl, nl, pos)
        sh = getattr(self, "_shard", None)
        if sh is not None and sh.world > 1:
            # data-parallel sequences: the reference's loss is the mean over the live positions of the WHOLE batch
            # (NN/trainers/sas.py:40-49).  Value: count-weighted mean of the ranks' means.  Gradient: this rank's share,
            # times the world size (GradSync averages the body gradients; the sharded table divides it out again).
            import torch.distributed as dist
            cnt = (pos != 0).sum().to(torch.float32).reshape(1)
            both = torch.cat([loss.detach().reshape(1) * cnt, cnt])
            dist.all_reduce(both, group=sh.group)
            share = loss * (cnt / both[1] * sh.world).reshape(())
            loss = (both[0] / both[1]).reshape(()) + (share - share.detach())
        return loss

    def last_hidden(self, log_seqs):
        if not self.training and not torch.is_grad_enabled():
            return self.log2feats(log_seqs, last_only=True)
        return self.log2feats(log_seqs)[:, -1, :]

    def predict(self, log_seqs, item_indices):  # for inference
        """NN/models/sas_model/sas.py:107-118 -> [B, C]."""
        if getattr(self, "_shard", None) is not None:
            from ..dist import sharded_candidate_scores
            return sharded_candidate_scores(self, log_seqs, item_indices)
        return ops.candidate_scores(self.last_hidden(log_seqs), self.sas.item_emb.weight, None, self._device_long(item_indices))

    def full_catalogue_topk(self, log_seqs, k=10, exclude=None):
        """Top-k items (ids 1..V), (score desc, id asc); the [B, V, d] gather of ``predict`` is never built (K19-K21).
        ``exclude`` ([B, n] int64 item ids, ids <= 0 = padding): items each user must not be ranked; ``exclude=log_seqs``
        ranks everything that is not in the input."""
        if getattr(self, "_shard", None) is not None:
            from ..dist import sharded_model_topk
            return sharded_model_topk(self, log_seqs, k, exclude=exclude)
        return ops.score_topk(self.last_hidden(log_seqs), self.sas.item_emb.weight, None, 1, self.sas.item_num + 1, k,
                              exclude=self._device_long(exclude) if exclude is not None else None)
