"""Shared pieces of the CPU oracle (TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py).

``NN/`` = ``/root/reference/NerualNetwork/bert4rec&sas4rec/``.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import numpy as np
import torch
import torch.nn.functional as F


class DropoutPlan:
    """How the oracle applies dropout at a named site.

    * ``p == 0`` or ``training == False``  -> identity (exact-parity mode).
    * ``masks`` given                      -> multiply by the supplied keep mask
      (uint8/bool, 1 = keep) and by 1/(1-p): the *injected-mask* mode used to
      compare training-mode CUDA kernels element-wise (the CUDA side exports
      the Philox mask it used for each site through ``rbm_dropout_mask``).
    * otherwise                            -> ``F.dropout`` exactly like the
      reference's ``nn.Dropout`` modules (used when timing the CPU baseline).
    """

    def __init__(self, training: bool = False, masks: Optional[Dict[int, torch.Tensor]] = None):
        self.training = training
        self.masks = masks

    def __call__(self, x: torch.Tensor, p: float, site: int) -> torch.Tensor:
        if not self.training or p == 0.0:
            return x
        if self.masks is not None:
            m = self.masks[site].to(x.dtype).reshape(x.shape)
            return x * m * (1.0 / (1.0 - p))
        return F.dropout(x, p=p, training=True)


NO_DROPOUT = DropoutPlan(training=False)


def _philox7(seed: int, site: int, call: np.ndarray):
    """Philox4x32-7 of the dropout sites: key = seed, counter = (call lo, call hi, site lo, site hi)."""
    from .batches import philox4x32
    call = np.asarray(call, dtype=np.uint64)
    return philox4x32((call, call >> np.uint64(32), site & 0xFFFFFFFF, site >> 32), (seed & 0xFFFFFFFF, seed >> 32), 7)


def keep_mask(n: int, p: float, seed: int, site: int) -> np.ndarray:
    """Keep mask (bool [n]) of an element-wise dropout site (include/rbm.h): element e takes word e % 4 of the Philox4x32-7 call
    e // 4 and is kept iff that word >= floor(p * 2^32), with p rounded to fp32 first as the C ABI passes it."""
    t = float(np.float32(p)) * 4294967296.0
    thr = 0 if t <= 0.0 else (0xFFFFFFFF if t >= 4294967295.0 else int(t))
    words = _philox7(seed, site, np.arange((n + 3) // 4, dtype=np.uint64))
    return (np.stack(words, axis=1).reshape(-1)[:n] >= thr)


def attn_keep_mask(BH: int, L: int, p: float, seed: int, site: int) -> np.ndarray:
    """Keep mask (bool [BH * L, L], row = bh * L + i, column = key j) of an attention dropout site (csrc/common.cuh): element
    (bh, i, j) is the 16-bit field  f = ((i >> 3) & 1) * 4 + (j & 1) * 2 + ((j >> 3) & 1)  (word f >> 1, high half when f is odd)
    of Philox4x32-7 call  ((((bh * 16 + (i >> 4)) * 8 + (i & 7)) * 4 + ((j & 7) >> 1)) * 16 + (j >> 4)),  kept iff the field
    >= round(p * 65536)."""
    t = float(np.float32(p)) * 65536.0 + 0.5
    thr16 = 0 if t <= 0.5 else (65535 if t >= 65535.0 else int(t))
    i = np.arange(L, dtype=np.int64)[:, None]
    j = np.arange(L, dtype=np.int64)[None, :]
    local = ((((i >> 4) * 8 + (i & 7)) * 4 + ((j & 7) >> 1)) * 16 + (j >> 4))  # the call index without bh: < 8192
    field = ((i >> 3) & 1) * 4 + (j & 1) * 2 + ((j >> 3) & 1)
    calls, inv = np.unique(local, return_inverse=True)
    inv = inv.reshape(L, L)
    bh = np.arange(BH, dtype=np.uint64)[:, None]
    words = np.stack(_philox7(seed, site, bh * np.uint64(8192) + calls.astype(np.uint64)[None, :]), axis=-1)  # [BH, calls, 4]
    w = words[:, inv, field >> 1]  # [BH, L, L]
    f16 = np.where((field & 1).astype(bool), w >> np.uint64(16), w & np.uint64(0xFFFF))
    return (f16 >= thr16).reshape(BH * L, L)


def torch_layernorm(x: torch.Tensor, w: torch.Tensor, b: torch.Tensor, eps: float) -> torch.Tensor:
    """``torch.nn.LayerNorm`` as used at NN/models/sas_model/sas.py:39,42,50 (eps=1e-8):
    biased variance, eps inside the sqrt."""
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) / torch.sqrt(var + eps) * w + b


def bert_layernorm(x: torch.Tensor, a_2: torch.Tensor, b_2: torch.Tensor, eps: float = 1e-6) -> torch.Tensor:
    """NN/models/bert_modules/utils/layer_norm.py:14-17 -- UNBIASED std (N-1), eps added to std."""
    mean = x.mean(-1, keepdim=True)
    std = x.std(-1, keepdim=True)
    return a_2 * (x - mean) / (std + eps) + b_2


def gelu_tanh(x: torch.Tensor) -> torch.Tensor:
    """NN/models/bert_modules/utils/gelu.py:12."""
    return 0.5 * x * (1 + torch.tanh(math.sqrt(2 / math.pi) * (x + 0.044715 * torch.pow(x, 3))))


def embedding_grad_scatter(idx: np.ndarray, rows: np.ndarray, vocab: int, padding_idx: int = 0) -> np.ndarray:
    """``embedding_dense_backward`` (autograd of nn.Embedding, NN/models/sas_model/sas.py:30,
    NN/models/bert_modules/embedding/token.py:6): grad[idx[i]] += rows[i] for i ascending;
    the ``padding_idx`` row receives nothing.  fp32 adds in index order -> this is the
    bit-exact contract of the sort/segment-reduce kernel."""
    idx = np.asarray(idx).reshape(-1)
    rows = np.asarray(rows, dtype=np.float32).reshape(idx.shape[0], -1)
    grad = np.zeros((vocab, rows.shape[1]), dtype=np.float32)
    for i in range(idx.shape[0]):
        t = int(idx[i])
        if t == padding_idx:
            continue
        grad[t] += rows[i]
    return grad


def embedding_grad_scatter_fast(idx: np.ndarray, rows: np.ndarray, vocab: int, padding_idx: int = 0) -> np.ndarray:
    """Same contract as :func:`embedding_grad_scatter` (np.add.at applies updates in element
    order), usable at sizes the python loop is too slow for."""
    idx = np.asarray(idx).reshape(-1)
    rows = np.asarray(rows, dtype=np.float32).reshape(idx.shape[0], -1)
    grad = np.zeros((vocab, rows.shape[1]), dtype=np.float32)
    keep = idx != padding_idx
    np.add.at(grad, idx[keep], rows[keep])
    return grad


def embedding_grad_scatter_chunked(idx: np.ndarray, rows: np.ndarray, vocab: int, padding_idx: int = 0,
                                   chunk: int = 64) -> np.ndarray:
    """The CUDA kernel's exact summation contract (rbm_scatter_add_sorted): per destination row the contributions,
    in ascending position, are cut into pieces of ``chunk``; each piece is summed sequentially, the piece sums are
    added in order.  Rows with <= chunk contributions coincide bit-for-bit with :func:`embedding_grad_scatter`
    (the reference's order); longer rows differ from it only in fp32 rounding."""
    idx = np.asarray(idx).reshape(-1)
    rows = np.asarray(rows, dtype=np.float32).reshape(idx.shape[0], -1)
    grad = np.zeros((vocab, rows.shape[1]), dtype=np.float32)
    order = np.argsort(idx, kind="stable")
    sidx = idx[order]
    bounds = np.flatnonzero(np.r_[True, sidx[1:] != sidx[:-1], True])
    for a, b in zip(bounds[:-1], bounds[1:]):
        key = int(sidx[a])
        if key == padding_idx:
            continue
        total = None
        for p0 in range(a, b, chunk):
            pos = order[p0:min(p0 + chunk, b)]
            acc = rows[pos[0]].copy()
            for r in pos[1:]:
                acc += rows[r]
            total = acc if total is None else total + acc
        grad[key] += total
    return grad


def synth_state_dict(shapes: Dict[str, tuple], seed: int, scale: float = 0.1) -> Dict[str, torch.Tensor]:
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randn(*s, generator=g) * scale for k, s in shapes.items()}
