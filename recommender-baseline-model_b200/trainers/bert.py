"""BERTTrainer -- task glue of NN/trainers/bert.py:8-52 over the fused kernels."""
import torch

from .base import AbstractTrainer
from .utils import full_catalogue_batch_metrics, recalls_ndcgs_and_mrr_for_ks


class BERTTrainer(AbstractTrainer):
    @classmethod
    def code(cls):
        return 'bert'

    def calculate_loss(self, batch):
        """NN/trainers/bert.py:30-41: CE(ignore_index=0) over the B*L x (V+1) logits -- computed by the fused
        scoring+CE kernel on the rows with labels != 0 only (identical value and gradients)."""
        seqs, labels = [x.to(self.device, non_blocking=True) for x in batch]
        return self.model.loss(seqs, labels)

    def calculate_metrics(self, batch):
        """NN/trainers/bert.py:43-52: last-position scores at the candidates -> Recall/NDCG/MRR@k.  With
        ``args.full_catalogue_eval`` the batch is (seq, answers, exclude) and every unseen item is ranked instead."""
        if getattr(self.args, 'full_catalogue_eval', False):
            return full_catalogue_batch_metrics(self.model, batch, self.metric_ks, self.device)
        seqs, candidates, labels = [x.to(self.device, non_blocking=True) for x in batch]
        scores = self.model.candidate_scores(seqs, candidates)
        return recalls_ndcgs_and_mrr_for_ks(scores, labels, self.metric_ks)
