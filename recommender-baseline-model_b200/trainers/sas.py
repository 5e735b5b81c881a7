"""SASTrainer -- task glue of NN/trainers/sas.py:9-62 over the fused kernels."""
import numpy as np
import torch

from .base import AbstractTrainer
from .utils import full_catalogue_batch_metrics, recalls_ndcgs_and_mrr_for_ks


class SASTrainer(AbstractTrainer):
    def __init__(self, args, model, train_loader, val_loader, test_loader, export_root):
        super().__init__(args, model, train_loader, val_loader, test_loader, export_root)
        self.l2_emb = args.l2_emb

    @classmethod
    def code(cls):
        return 'sas'

    def close_training(self):
        if hasattr(self.train_loader, 'close'):
            self.train_loader.close()

    def calculate_loss(self, batch):
        """NN/trainers/sas.py:34-54: BCE(pos,1)+BCE(neg,0) over pos != 0, plus l2_emb * sum ||param||_2."""
        seq, pos, neg = batch
        if not torch.is_tensor(seq):
            seq, pos, neg = np.array(seq), np.array(pos), np.array(neg)
        loss = self.model.loss(seq, pos, neg)
        if self.l2_emb != 0.0:
            for param in self.model.parameters():
                loss = loss + self.l2_emb * torch.norm(param)
        return loss

    def calculate_metrics(self, batch):
        """NN/trainers/sas.py:56-62.  With ``args.full_catalogue_eval`` the batch is (seq, answers, exclude) and every unseen item
        is ranked instead."""
        if getattr(self.args, 'full_catalogue_eval', False):
            return full_catalogue_batch_metrics(self.model, batch, self.metric_ks, self.device)
        seqs, candidates, labels = batch
        logits = self.model.predict(seqs, candidates)
        return recalls_ndcgs_and_mrr_for_ks(logits, labels, self.metric_ks)
