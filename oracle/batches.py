"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): CPU restatement of the reference's training-batch construction.

Follows ``BertTrainDataset.__getitem__`` (NN/dataloaders/bert.py:77-110) and ``sample_function`` / ``random_neq``
(NN/dataloaders/sas.py:65-86), NN/ = NerualNetwork/bert4rec&sas4rec/.  The reference draws from numpy's global /
RandomState streams, which no device kernel can reproduce; like dropout, the random numbers are therefore part of the
contract: Philox4x32-10 (Salmon et al., SC'11; restated below and pinned against the Random123 known-answer vectors in
tests/test_oracle_golden.py) with key = seed and counter = (idx4, site), consumed exactly as written in
include/rbm.h / csrc/batch.cu.  Given those numbers every branch below is the reference's.
"""
import math
from typing import List, Sequence, Tuple

import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = 0xFFFFFFFF


def philox4x32(counter: Sequence, key: Sequence[int], rounds: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """Philox4x32 with ``rounds`` rounds over numpy arrays: counter words (c0..c3, each an int or an array; they broadcast
    against each other), key (k0, k1) -> four uint64 arrays holding the 32-bit output words."""
    c0, c1, c2, c3 = [np.asarray(c, dtype=np.uint64) & np.uint64(MASK32) for c in counter]
    k0, k1 = [int(k) & MASK32 for k in key]
    m0, m1, lo32 = np.uint64(M0), np.uint64(M1), np.uint64(MASK32)
    for _ in range(rounds):
        p0, p1 = m0 * c0, m1 * c2  # 32 x 32 -> 64 bits: exact in uint64
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & lo32, p1 >> np.uint64(32), p1 & lo32
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0
        k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
    return c0, c1, c2, c3


def philox4x32_10(counter: Sequence[int], key: Sequence[int]) -> Tuple[int, int, int, int]:
    """One Philox4x32-10 block: counter (c0..c3), key (k0, k1) -> four 32-bit words."""
    return tuple(int(w) for w in philox4x32(counter, key, 10))


def rbm_philox(seed: int, site: int, idx4: int) -> Tuple[int, int, int, int]:
    """The library's call convention: counter = (idx4 lo, idx4 hi, site lo, site hi), key = (seed lo, seed hi)."""
    return philox4x32_10((idx4 & MASK32, idx4 >> 32, site & MASK32, site >> 32), (seed & MASK32, seed >> 32))


def bert_cloze_batch(histories: List[List[int]], users: Sequence[int], max_len: int, mask_prob: float, mask_token: int,
                     num_items: int, seed: int, site: int) -> Tuple[np.ndarray, np.ndarray]:
    """bert.py:77-110 -- for every item of the (truncated, :100-101) sequence: prob < mask_prob -> label = item and token =
    [MASK] if prob/mask_prob < 0.8, a uniform item of 1..num_items if < 0.9, else itself (:84-95); otherwise token = item,
    label = 0 (:96-98); left padding with 0 (:103-108)."""
    X = mask_prob * 4294967296.0  # prob = u / 2^32:  prob < p  <=>  u < ceil(X);  prob/p < 0.8  <=>  u < ceil(0.8 X) ...
    thr, t80, t90 = math.ceil(X), math.ceil(0.8 * X), math.ceil(0.9 * X)
    B = len(users)
    tokens = np.zeros((B, max_len), np.int64)
    labels = np.zeros((B, max_len), np.int64)
    for b, u in enumerate(users):
        seq = list(histories[u])[-max_len:]
        pad = max_len - len(seq)
        for k, s in enumerate(seq):
            p = pad + k
            r = rbm_philox(seed, site, b * 128 + (p >> 1))
            dec, w = r[2 * (p & 1)], r[2 * (p & 1) + 1]
            tok, lab = s, 0
            if dec < thr:
                lab = s
                if dec < t80:
                    tok = mask_token
                elif dec < t90:
                    tok = 1 + ((w * num_items) >> 32)
            tokens[b, p], labels[b, p] = tok, lab
    return tokens, labels


def sas_train_batch(histories: List[List[int]], users: Sequence[int], max_len: int, num_items: int, seed: int,
                    site: int) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """sas.py:65-86 -- train = history[-max_len:]; padding_len = max_len - len(train) + 1; seq = pad + train[:-1];
    pos = pad + train[1:]; neg = pad + random_neq(0, item_num, set(train), len(train) - 1), i.e. a uniform pick from the
    (ascending) list of ids in [0, item_num] outside the window -- id 0 included, as in the reference."""
    B = len(users)
    seq = np.zeros((B, max_len), np.int64)
    pos = np.zeros((B, max_len), np.int64)
    neg = np.zeros((B, max_len), np.int64)
    for b, u in enumerate(users):
        train = list(histories[u])[-max_len:]
        if len(train) < 2:
            continue
        pad = max_len - len(train) + 1
        a = sorted(set(range(0, num_items + 1)) - set(train))
        for k in range(len(train) - 1):
            p = pad + k
            seq[b, p], pos[b, p] = train[k], train[k + 1]
            if a:
                r = rbm_philox(seed, site, b * 64 + (p >> 2))
                neg[b, p] = a[(r[p & 3] * len(a)) >> 32]
    return seq, pos, neg


NEG_MAX_ATTEMPTS = 65536


def negative_samples(seen: List[Sequence[int]], num_items: int, n_samples: int, seed: int, site: int,
                     pop_counts: Sequence[int] = None, user_begin: int = 0, num_users: int = None) -> np.ndarray:
    """Evaluation negatives (NN/dataloaders/negative_samplers/random.py:13-37, popular.py:15-44) with the contract's numbers:
    attempt t of user u draws r64 from Philox call u * 65536 + t (words 0, 1); uniform: item = 1 + (r64 * V >> 64)
    (random.py:29, ``np.random.choice(item_count) + 1``); popularity: x = r64 * total >> 64, item = first id whose inclusive
    count prefix sum exceeds x (popular.py:18-22,33: p = count / total).  An attempt is kept unless the item is in the user's
    seen set (random.py:30, popular.py:34) or already kept; the first ``n_samples`` kept items are the row.
    ``pop_counts[i]`` = interaction count of item i + 1."""
    U = len(seen) - user_begin if num_users is None else num_users
    out = np.full((U, n_samples), -1, np.int64)
    cdf = None if pop_counts is None else np.cumsum(np.asarray(pop_counts, dtype=object))
    for row in range(U):
        u = user_begin + row
        s, got = set(int(i) for i in seen[u]), []
        for t in range(NEG_MAX_ATTEMPTS):
            if len(got) == n_samples:
                break
            r = rbm_philox(seed, site, u * NEG_MAX_ATTEMPTS + t)
            r64 = (r[0] << 32) | r[1]
            if cdf is None:
                item = 1 + ((r64 * num_items) >> 64)
            else:
                x = (r64 * int(cdf[-1])) >> 64
                item = 1 + next(i for i in range(num_items) if cdf[i] > x)
            if item in s or item in got:
                continue
            got.append(item)
        out[row, :len(got)] = got
    return out


def eval_batch(histories: List[Sequence[int]], answers: Sequence[int], negatives: np.ndarray, users: Sequence[int], max_len: int,
               mask_token: int = -1) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """BertEvalDataset.__getitem__ (NN/dataloaders/bert.py:128-142: seq + [mask_token], last max_len, left pad) /
    SASEvalDataset.__getitem__ (NN/dataloaders/sas.py:136-153: no mask token, ``mask_token = -1`` here);
    candidates = answer + negatives, labels = [1] + [0] * n."""
    B, n_neg = len(users), negatives.shape[1]
    seq = np.zeros((B, max_len), np.int64)
    cand = np.zeros((B, 1 + n_neg), np.int64)
    labels = np.zeros((B, 1 + n_neg), np.int64)
    for b, u in enumerate(users):
        s = list(histories[u]) + ([mask_token] if mask_token >= 0 else [])
        s = s[-max_len:]
        if s:
            seq[b, max_len - len(s):] = s
        cand[b, 0], cand[b, 1:] = answers[u], negatives[u]
        labels[b, 0] = 1
    return seq, cand, labels
