"""ctypes binding of librbm_b200.so (the C ABI declared in include/rbm.h).

There is NO fallback: if the library is missing or a call fails, a RuntimeError is raised.  Tensors are passed as
raw device pointers; kernels run on torch's current CUDA stream; scratch memory comes from torch's allocator.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, Optional

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librbm_b200.so")
HEADER = os.path.join(os.path.dirname(HERE), "include", "rbm.h")

ACT_NONE, ACT_RELU, ACT_GELU_TANH = 0, 1, 2
LN_TORCH, LN_BERT = 0, 1
MASK_NONE, MASK_CAUSAL, MASK_KEYPAD = 0, 1, 2
ADAM_CHUNK = 4096

_P, _I, _L, _F, _D, _U64, _SZ = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_uint64, C.c_size_t

# name -> (restype, argtypes); must list every function include/rbm.h declares (tests/test_abi.py checks this)
SIGNATURES = {
    "rbm_abi_version": (_I, []),
    "rbm_last_error": (C.c_char_p, []),
    "rbm_embed_fwd": (_I, [_P, _P, _P, _P, _L, _I, _I, _L, _F, _I, _F, _U64, _U64, _P]),
    "rbm_embed_bwd": (_I, [_P, _P, _P, _P, _L, _I, _I, _I, _F, _U64, _U64, _P]),
    "rbm_embed_fwd_shard": (_I, [_P, _P, _P, _P, _L, _I, _I, _L, _L, _L, _F, _I, _F, _U64, _U64, _P]),
    "rbm_embed_bwd_offset": (_I, [_P, _P, _P, _P, _L, _I, _I, _I, _F, _U64, _U64, _U64, _P]),
    "rbm_scatter_ws_bytes": (_SZ, [_L, _L]),
    "rbm_scatter_add_sorted": (_I, [_P, _P, _P, _F, _P, _L, _I, _L, _L, _P, _SZ, _P]),
    "rbm_layernorm_fwd": (_I, [_P, _P, _P, _P, _P, _L, _I, _F, _I, _P]),
    "rbm_layernorm_ws_bytes": (_SZ, [_L, _I]),
    "rbm_layernorm_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _I, _P, _SZ, _P]),
    "rbm_layernorm_bwd_residual": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _I, _P, _SZ, _P]),
    "rbm_layernorm_bwd_fanout": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _I, _P, _SZ, _P]),
    "rbm_linear_fwd": (_I, [_P, _L, _P, _P, _P, _L, _P, _L, _I, _I, _I, _P, _L, _P, _F, _U64, _F, _U64, _U64, _P]),
    "rbm_linear_fwd_ws_bytes": (_SZ, [_L, _I, _I]),
    "rbm_linear_fwd_ws": (_I, [_P, _L, _P, _P, _P, _L, _P, _L, _I, _I, _I, _P, _L, _P, _F, _U64, _F, _U64, _U64, _P, _SZ, _P]),
    "rbm_linear_epilogue_bwd": (_I, [_P, _P, _P, _P, _L, _I, _I, _P, _F, _U64, _F, _U64, _U64, _P]),
    "rbm_linear_bwd_data_ws_bytes": (_SZ, [_I, _I]),
    "rbm_linear_bwd_data": (_I, [_P, _L, _P, _P, _L, _L, _I, _I, _P, _SZ, _P]),
    "rbm_linear_bwd_weight_ws_bytes": (_SZ, [_L, _I, _I]),
    "rbm_linear_bwd_weight": (_I, [_P, _L, _P, _L, _P, _P, _L, _I, _I, _P, _SZ, _P]),
    "rbm_embed_bwd_rows_ws_bytes": (_SZ, [_I, _I]),
    "rbm_embed_bwd_rows": (_I, [_P, _P, _P, _L, _P, _P, _P, _P, _I, _I, _F, _U64, _U64, _P, _SZ, _P]),
    "rbm_rows_gather": (_I, [_P, _L, _P, _P, _L, _I, _P, _P, _P]),
    "rbm_rows_scatter": (_I, [_P, _P, _P, _L, _I, _P, _P, _L, _P, _L, _P]),
    "rbm_rows_dead_colsum_ws_bytes": (_SZ, [_I]),
    "rbm_rows_dead_colsum": (_I, [_P, _L, _P, _L, _I, _P, _P, _SZ, _P]),
    "rbm_rows_live_colsum": (_I, [_P, _L, _P, _L, _I, _P, _P, _SZ, _P]),
    "rbm_rows_seq_start": (_I, [_P, _P, _I, _I, _P, _P]),
    "rbm_attn_live_fwd": (_I, [_P, _L, _P, _L, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _F, _U64, _U64, _P]),
    "rbm_attn_live_bwd": (_I, [_P, _L, _P, _L, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _F, _U64, _U64, _P]),
    "rbm_rows_to_seq": (_I, [_P, _P, _I, _I, _I, _P, _P]),
    "rbm_seq_to_rows": (_I, [_P, _P, _P, _P, _L, _I, _I, _I, _P, _P]),
    "rbm_attn_lq_supported": (_I, [_I, _I, _I, _I]),
    "rbm_attn_fwd_lq": (_I, [_P, _L, _P, _L, _P, _L, _P, _P, _L, _P, _I, _I, _I, _I, _I, _I, _F, _F, _U64, _U64, _P]),
    "rbm_attn_bwd_lq_ws_bytes": (_SZ, [_I, _I, _I]),
    "rbm_attn_bwd_lq": (_I, [_P, _L, _P, _L, _P, _L, _P, _P, _L, _P, _L, _P, _P, _L, _P, _L, _P, _L, _I, _I, _I, _I, _I, _I, _F,
                             _F, _U64, _U64, _P, _SZ, _P]),
    "rbm_attn_last_query": (_I, [_P, _L, _P, _L, _P, _L, _P, _P, _L, _I, _I, _I, _I, _I, _F, _P]),
    "rbm_attn_fwd": (_I, [_P, _L, _P, _L, _P, _L, _P, _P, _L, _P, _I, _I, _I, _I, _I, _F, _F, _U64, _U64, _P]),
    "rbm_attn_bwd_ws_bytes": (_SZ, [_I, _I, _I]),
    "rbm_attn_bwd": (_I, [_P, _L, _P, _L, _P, _L, _P, _P, _L, _P, _L, _P, _P, _L, _P, _L, _P, _L, _I, _I, _I, _I, _I, _F,
                          _F, _U64, _U64, _P, _SZ, _P]),
    "rbm_compact_ws_bytes": (_SZ, [_L]),
    "rbm_compact_labels": (_I, [_P, _L, _P, _P, _P, _P, _SZ, _P]),
    "rbm_ce_ws_bytes": (_SZ, [_L, _I, _I]),
    "rbm_ce_fwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _P, _SZ, _P]),
    "rbm_ce_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _I, _I, _P, _SZ, _P]),
    "rbm_sas_score_fwd": (_I, [_P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "rbm_sas_score_bwd": (_I, [_P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "rbm_bce_ws_bytes": (_SZ, [_L]),
    "rbm_bce_pair_fwd": (_I, [_P, _P, _P, _P, _P, _L, _P, _SZ, _P]),
    "rbm_bce_pair_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _P]),
    "rbm_candidate_scores": (_I, [_P, _L, _P, _P, _P, _P, _L, _I, _I, _P]),
    "rbm_score_topk_ws_bytes": (_SZ, [_L, _L, _I]),
    "rbm_score_topk_ws_bytes_d": (_SZ, [_L, _L, _I, _I]),
    "rbm_score_topk": (_I, [_P, _L, _P, _P, _L, _L, _L, _P, _P, _L, _I, _I, _P, _SZ, _P]),
    "rbm_score_topk_excl": (_I, [_P, _L, _P, _P, _L, _L, _L, _P, _L, _I, _P, _P, _L, _I, _I, _P, _SZ, _P]),
    "rbm_topk_rows": (_I, [_P, _L, _P, _P, _L, _L, _I, _L, _P]),
    "rbm_topk_merge": (_I, [_P, _P, _P, _P, _I, _L, _I, _P]),
    "rbm_rank_metrics": (_I, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _I, _L, _L, _P]),
    "rbm_column_mean_ws_bytes": (_SZ, [_L, _I]),
    "rbm_column_mean": (_I, [_P, _P, _L, _I, _P, _SZ, _P]),
    "rbm_adam_multi": (_I, [_P, _P, _I, _D, _D, _D, _D, _D, _I, _P]),
    "rbm_bucket_pack": (_I, [_P, _P, _I, _P, _F, _I, _P]),
    "rbm_set_step_counter": (_I, [_P]),
    "rbm_bert_cloze_batch": (_I, [_P, _P, _P, _I, _I, _D, _L, _L, _U64, _U64, _P, _P, _P]),
    "rbm_sas_train_batch": (_I, [_P, _P, _P, _I, _I, _L, _U64, _U64, _P, _P, _P, _P]),
    "rbm_negative_samples": (_I, [_P, _P, _P, _L, _L, _L, _I, _U64, _U64, _P, _P]),
    "rbm_eval_batch": (_I, [_P, _P, _P, _P, _P, _I, _I, _I, _L, _P, _P, _P, _P]),
    "rbm_dropout_mask": (_I, [_P, _L, _F, _U64, _U64, _P]),
    "rbm_dropout_mask_attn": (_I, [_P, _L, _I, _F, _U64, _U64, _P]),
}

_lib: Optional[C.CDLL] = None


def header_functions():
    """Names of every function declared in include/rbm.h."""
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(rbm_[a-z0-9_]+)\s*\(", src)))


def load() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built -- there is no CPU / torch fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "librbm_b200.so is missing (%s). Build it with `python __graft_entry__.py build` "
            "(nvcc, sm_100a). This package has no CPU or PyTorch fallback." % LIB_PATH)
    cdll = C.CDLL(LIB_PATH)
    lib = _Lib()
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(cdll, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
        setattr(lib, name, _timed(name, fn) if res is _I and name != "rbm_abi_version" else fn)
    if lib.rbm_abi_version() != 1:
        raise RuntimeError("librbm_b200.so ABI version mismatch")
    _lib = lib
    return lib


class _Lib:
    """Namespace of the bound C functions."""


# Optional per-entry-point device timing (bench.py's roofline leg): when `profile` is a dict, every kernel-launching
# call is bracketed by CUDA events on the launching stream; `profile_collect()` turns them into milliseconds.
profile = None


def _timed(name, fn):
    def call(*a):
        if profile is None:
            return fn(*a)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*a)
        e1.record()
        profile.setdefault(name, []).append((e0, e1, a))
        return rc
    return call


def profile_collect():
    """{entry point: [(ms, call args)]} for the calls recorded since `profile` was set to a dict."""
    torch.cuda.synchronize()
    return {k: [(a.elapsed_time(b), args) for a, b, args in v] for k, v in (profile or {}).items()}


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().rbm_last_error().decode("utf-8", "replace")
        raise RuntimeError("librbm_b200 %s failed (rc=%d): %s" % (what, rc, msg))


def ptr(t: Optional[torch.Tensor]):
    if t is None:
        return None
    return t.data_ptr()


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors: torch.Tensor):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("rbm_b200 ops run on CUDA tensors only (got a %s tensor): there is no CPU fallback" % t.device)


class _Workspaces:
    """Grow-only scratch buffers per (device, tag); reuse is safe because every consumer is stream-ordered.  A captured CUDA
    graph has the buffer addresses baked into its kernel nodes: while any graph is alive (``freeze`` / ``unfreeze``, called by
    ``capture_train_step`` / ``release_train_graph``) a buffer that has to grow is retired, not freed, so replays keep
    writing into memory that is still theirs."""

    def __init__(self):
        self.bufs: Dict[tuple, torch.Tensor] = {}
        self.frozen = 0
        self.retired = []

    def freeze(self):
        self.frozen += 1

    def unfreeze(self):
        self.frozen = max(0, self.frozen - 1)
        if self.frozen == 0:
            self.retired.clear()

    def get(self, tag: str, nbytes: int, device) -> torch.Tensor:
        key = (str(device), tag)
        buf = self.bufs.get(key)
        if buf is None or buf.numel() < nbytes:
            if buf is not None and self.frozen:
                self.retired.append(buf)
            buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
            self.bufs[key] = buf
        return buf


workspaces = _Workspaces()

# number of kernels of this library launched since the last reset (bench.py reports it as gpu_launches)
launch_count = 0


def count_launches(n: int = 1):
    global launch_count
    launch_count += n
