"""Training-batch producers that run ON THE DEVICE (SURVEY.md 8(f) #1).

The reference builds every batch with python per-item loops, ``deepcopy`` and (SASRec) ``multiprocessing.Queue`` pickling
(NN/dataloaders/bert.py:77-110, NN/dataloaders/sas.py:65-114).  Here the user histories live on the GPU as a CSR and a
batch is one kernel launch (``rbm_bert_cloze_batch`` / ``rbm_sas_train_batch``); what comes out has the reference's wire
format (int64 ``[B, L]`` tensors, left-padded with 0), so the trainers consume it unchanged.  A batch is a pure function
of (histories, users, seed, step): the Philox field layout is part of the C-ABI contract (include/rbm.h)."""
from typing import Dict, Sequence, Union

import numpy as np
import torch

from .. import ops


def histories_to_csr(user_train: Union[Dict[int, Sequence[int]], Sequence[Sequence[int]]], device):
    """``user_train`` of ``data_partition`` (dict user -> item list, or a list of lists) -> (hist_ptr, hist_items) on device."""
    rows = [user_train[u] for u in sorted(user_train)] if isinstance(user_train, dict) else list(user_train)
    ptr = np.zeros(len(rows) + 1, np.int64)
    np.cumsum([len(r) for r in rows], out=ptr[1:])
    items = np.fromiter((i for r in rows for i in r), np.int64, count=int(ptr[-1]))
    return torch.from_numpy(ptr).to(device), torch.from_numpy(items).to(device)


class DeviceBertTrainLoader:
    """Epoch iterator of ``(tokens, labels)`` like ``DataLoader(BertTrainDataset, shuffle=True)`` (NN/dataloaders/bert.py:25-34)."""

    def __init__(self, user_train, max_len: int, mask_prob: float, num_items: int, batch_size: int, device, seed: int = 0):
        self.ptr, self.items = histories_to_csr(user_train, device)
        self.num_users = self.ptr.numel() - 1
        self.max_len, self.mask_prob, self.num_items, self.batch_size = max_len, mask_prob, num_items, batch_size
        self.mask_token = num_items + 1
        self.seed, self.step = seed, 0
        self.gen = torch.Generator(device=device)
        self.gen.manual_seed(seed)

    def __len__(self):
        return (self.num_users + self.batch_size - 1) // self.batch_size

    def __iter__(self):
        perm = torch.randperm(self.num_users, device=self.ptr.device, generator=self.gen)
        for b in range(len(self)):
            users = perm[b * self.batch_size:(b + 1) * self.batch_size].contiguous()
            yield ops.bert_cloze_batch(self.ptr, self.items, users, self.max_len, self.mask_prob, self.mask_token, self.num_items,
                                       self.seed, self.step)
            self.step += 1


class DeviceSasTrainLoader:
    """``WarpSampler`` (NN/dataloaders/sas.py:92-121): ``len(user_train) // batch_size`` batches per epoch, every row a uniformly
    drawn user (with replacement), as ``(seq, pos, neg)`` device tensors."""

    def __init__(self, user_train, max_len: int, num_items: int, batch_size: int, device, seed: int = 0):
        self.ptr, self.items = histories_to_csr(user_train, device)
        self.num_users = self.ptr.numel() - 1
        self.max_len, self.num_items, self.batch_size = max_len, num_items, batch_size
        self.seed, self.step = seed, 0
        self.gen = torch.Generator(device=device)
        self.gen.manual_seed(seed)

    def __len__(self):
        return self.num_users // self.batch_size

    def __iter__(self):
        for _ in range(len(self)):
            users = torch.randint(0, self.num_users, (self.batch_size,), device=self.ptr.device, generator=self.gen)
            yield ops.sas_train_batch(self.ptr, self.items, users, self.max_len, self.num_items, self.seed, self.step)
            self.step += 1


def seen_sets_to_csr(*splits, device):
    """Union of each user's items over the given splits (train, val, test as ``data_partition`` returns them), ascending and
    unique, as a CSR on the device -- the ``seen`` sets of the reference's negative samplers (random.py:25-27, popular.py:27-29)."""
    first = splits[0]
    users = sorted(first) if isinstance(first, dict) else range(len(first))
    rows = [np.unique(np.fromiter((i for s in splits for i in s[u]), np.int64)) for u in users]
    ptr = np.zeros(len(rows) + 1, np.int64)
    np.cumsum([len(r) for r in rows], out=ptr[1:])
    items = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    return torch.from_numpy(ptr).to(device), torch.from_numpy(items).to(device)


def popularity_cdf(num_items: int, *splits, device):
    """Inclusive prefix sums (int64 [num_items]) of the interaction counts of items 1..num_items over the given splits
    (``items_by_popularity``, NN/dataloaders/negative_samplers/popular.py:46-53)."""
    first = splits[0]
    users = sorted(first) if isinstance(first, dict) else range(len(first))
    counts = np.zeros(num_items + 1, np.int64)
    for s in splits:
        for u in users:
            np.add.at(counts, np.asarray(s[u], np.int64), 1)
    return torch.from_numpy(np.cumsum(counts[1:])).to(device)


class DeviceNegativeSampler:
    """``negative_sampler_factory(code, ...).get_negative_samples()`` on the device (NN/dataloaders/negative_samplers/):
    ``code`` 'random' (uniform) or 'popular' (interaction-count weighted); ``sample_size`` distinct unseen items per user as one
    ``[U, sample_size]`` int64 tensor (row u = the reference's ``negative_samples[u]``).  Raises if a user has fewer than
    ``sample_size`` unseen items to draw from (the reference would loop forever)."""

    def __init__(self, train, val, test, user_count: int, item_count: int, sample_size: int, seed: int, device, code: str = "random"):
        if code not in ("random", "popular"):
            raise ValueError("negative sampler code must be 'random' or 'popular'")
        if seed is None:
            raise AssertionError("Specify seed for random sampling")  # random.py:14
        self.code, self.item_count, self.sample_size, self.seed = code, item_count, sample_size, int(seed)
        self.seen_ptr, self.seen_items = seen_sets_to_csr(train, val, test, device=device)
        if self.seen_ptr.numel() - 1 != user_count:
            raise ValueError("user_count does not match the splits")
        self.cdf = popularity_cdf(item_count, train, val, test, device=device) if code == "popular" else None

    def get_negative_samples(self) -> torch.Tensor:
        out = ops.negative_samples(self.seen_ptr, self.seen_items, self.item_count, self.sample_size, self.seed, self.cdf)
        if bool((out < 0).any()):
            raise RuntimeError("negative sampling: some user has fewer than sample_size unseen items within reach")
        return out


class DeviceEvalLoader:
    """``DataLoader(BertEvalDataset | SASEvalDataset, shuffle=False)`` (NN/dataloaders/bert.py:44-62,116-142, sas.py:49-62,124-153):
    batches of ``(seq, candidates, labels)`` device tensors in user order; ``mask_token`` = V+1 for BERT4Rec (appended to the
    history before the cut to ``max_len``), -1 for SASRec.  ``history`` is what the reference passes as ``u2seq`` (train for
    validation; train ++ val for the test split of the 'leave one out' protocol), ``answers`` one held-out item per user.

    ``full_catalogue=True`` (full-ranking protocol; ``negatives`` unused): batches of ``(seq [B, L], answers [B],
    exclude [B, n])`` instead, where row u of ``exclude`` is user u's whole history (not only its last ``max_len`` items), zero-
    padded to the batch's longest, with the user's own answer removed so that an item the user returns to stays rankable."""

    def __init__(self, history, answers, negatives: torch.Tensor, max_len: int, batch_size: int, device, mask_token: int = -1,
                 full_catalogue: bool = False):
        self.ptr, self.items = histories_to_csr(history, device)
        self.num_users = self.ptr.numel() - 1
        users = sorted(answers) if isinstance(answers, dict) else range(len(answers))
        ans = [answers[u][0] if isinstance(answers[u], (list, tuple, np.ndarray)) else answers[u] for u in users]
        self.answers = torch.tensor(ans, dtype=torch.int64, device=device)
        self.full_catalogue = bool(full_catalogue)
        self.negatives = None if (negatives is None or self.full_catalogue) else negatives.to(device).contiguous()
        self.max_len, self.batch_size, self.mask_token = max_len, batch_size, mask_token
        # row lengths on the host: the width of a batch's exclusion matrix is known without a device round trip
        self.lengths = self.ptr.diff().cpu().numpy() if self.full_catalogue else None

    def __len__(self):
        return (self.num_users + self.batch_size - 1) // self.batch_size

    def _exclude(self, b0: int, b1: int, answers: torch.Tensor) -> torch.Tensor:
        """The histories of users [b0, b1) as a zero-padded [b1 - b0, n] matrix (their CSR rows are one contiguous slice)."""
        n = int(self.lengths[b0:b1].max()) if b1 > b0 else 0
        dev = self.ptr.device
        if n == 0:
            return torch.zeros(b1 - b0, 0, device=dev, dtype=torch.int64)
        start = self.ptr[b0:b1].unsqueeze(1)
        col = torch.arange(n, device=dev, dtype=torch.int64).unsqueeze(0)
        valid = col < (self.ptr[b0 + 1:b1 + 1].unsqueeze(1) - start)
        ex = torch.where(valid, self.items[(start + col).clamp_max(self.items.numel() - 1)], 0)
        return ex.masked_fill_(ex == answers.unsqueeze(1), 0)

    def __iter__(self):
        for b in range(len(self)):
            b0, b1 = b * self.batch_size, min((b + 1) * self.batch_size, self.num_users)
            users = torch.arange(b0, b1, device=self.ptr.device)
            seq, cand, labels = ops.eval_batch(self.ptr, self.items, self.answers, self.negatives, users, self.max_len, self.mask_token)
            if self.full_catalogue:
                answers = self.answers[b0:b1]
                yield seq, answers, self._exclude(b0, b1, answers)
            else:
                yield seq, cand, labels
