"""``recalls_ndcgs_and_mrr_for_ks`` -- NN/trainers/utils.py:28-57 on the GPU.

The reference copies all scores to the host and fully sorts every row; here a top-max(ks) selection kernel
(score desc, index asc -- the canonical form of its unstable argsort), a per-user metric kernel and a fixed-order
mean run on the device, and only the 3*len(ks) means come back."""
from __future__ import annotations

import torch

from .. import ops


def _as_dict(ks, means):
    out = {}
    for j, k in enumerate(ks):
        out['Recall@%d' % k] = means[j * 3 + 0]
        out['NDCG@%d' % k] = means[j * 3 + 1]
        out['MRR@%d' % k] = means[j * 3 + 2]
    return out


def recalls_ndcgs_and_mrr_for_ks(scores, labels, ks):
    """scores [B,C] f32, labels [B,C] i64 (1 = relevant) -> {'Recall@k','NDCG@k','MRR@k': float} batch means."""
    ks = sorted(int(k) for k in ks)[::-1]
    if not scores.is_cuda:
        raise RuntimeError("recalls_ndcgs_and_mrr_for_ks: scores must live on the GPU (no CPU fallback)")
    labels = labels.to(device=scores.device, dtype=torch.long)
    K = max(ks)
    if K > 32:
        raise RuntimeError("metric cut-offs above 32 are not supported by the top-k kernel (got %d)" % K)
    _, top_ids = ops.topk_rows(scores, K)
    per_user = ops.rank_metrics(top_ids, ks, labels=labels)
    means = ops.column_mean(per_user).tolist()
    return _as_dict(ks, means)


def full_catalogue_metrics(top_ids, positives, ks):
    """HR/NDCG/MRR@k of a full-catalogue top-K list against one held-out positive per user (batch means)."""
    ks = sorted(int(k) for k in ks)[::-1]
    per_user = ops.rank_metrics(top_ids, ks, positives=positives.to(device=top_ids.device, dtype=torch.long))
    means = ops.column_mean(per_user).tolist()
    return _as_dict(ks, means)


def full_catalogue_batch_metrics(model, batch, ks, device):
    """Metrics of one ``(seq, answers, exclude)`` batch of the full-catalogue protocol (``args.full_catalogue_eval``): each user's
    answer ranked among ALL items minus ``exclude`` (their history), same keys as the sampled protocol.  max(ks) <= 10 runs the
    tcgen05 selection path; 11..32 the exact fp32 scan, which is exact but slow at 10^7 items."""
    K = max(int(k) for k in ks)
    if K > 32:
        raise RuntimeError("metric cut-offs above 32 are not supported by the top-k kernel (got %d)" % K)
    seqs, answers, exclude = [x.to(device, non_blocking=True) for x in batch]
    _, top_ids = model.full_catalogue_topk(seqs, K, exclude=exclude)
    return full_catalogue_metrics(top_ids, answers, ks)
