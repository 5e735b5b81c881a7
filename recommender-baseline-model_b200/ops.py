"""autograd.Functions over the C ABI (include/rbm.h).  Each op = one group of reference torch ops replaced by a
hand-written sm_100a kernel; `loss.backward()` (NN/trainers/base.py:121) walks these backward methods.
No torch math on the hot path: torch only allocates the output tensors and orders the calls."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import lib as L
from .lib import check, ptr, stream, workspaces, count_launches


def _ws(tag: str, nbytes: int, device) -> torch.Tensor:
    return workspaces.get(tag, nbytes, device)


def _rows2d(x: torch.Tensor) -> torch.Tensor:
    """View as [rows, cols] with unit inner stride (no copy when already so)."""
    x2 = x.reshape(-1, x.shape[-1])
    if x2.stride(-1) != 1:
        x2 = x2.contiguous()
    return x2


# ------------------------------------------------------------------------------------------ scatter-add
def scatter_add_sorted_(grad: torch.Tensor, idx: torch.Tensor, src: torch.Tensor, coef: Optional[torch.Tensor] = None,
                        alpha: float = 1.0, padding_idx: int = 0, vocab: Optional[int] = None) -> torch.Tensor:
    """grad[idx[i]] += alpha*coef[i]*src[i] in ascending i per row (deterministic; K17).  ``vocab`` (default: rows of ``grad``)
    bounds the keys; a key range one larger than ``grad`` with ``padding_idx = grad.shape[0]`` gives a skip key that is not a row."""
    lib = L.load()
    L.require_cuda(grad, idx, src)
    n, d = idx.numel(), grad.shape[1]
    idx = idx.reshape(-1).contiguous()
    src = src.reshape(n, d).contiguous()
    vocab = grad.shape[0] if vocab is None else int(vocab)
    if vocab > grad.shape[0] and not (vocab == grad.shape[0] + 1 and padding_idx == grad.shape[0]):
        raise RuntimeError("scatter_add_sorted_: keys beyond the rows of grad must be the skipped padding key")
    nb = lib.rbm_scatter_ws_bytes(n, vocab)
    ws = _ws("scatter", nb, grad.device)
    check(lib.rbm_scatter_add_sorted(ptr(idx), ptr(src), ptr(coef), float(alpha), ptr(grad), n, d, vocab,
                                     int(padding_idx), ptr(ws), nb, stream()), "scatter_add_sorted")
    bits = max(1, (vocab - 1).bit_length())
    count_launches(3 * ((bits + 7) // 8) + 2)
    return grad


# ------------------------------------------------------------------------------------- live-row compaction (SASRec)
class LiveRows:
    """The live (token != 0) rows of a [B, L] batch: ascending row ids + count on the device (rbm_compact_labels applied to the
    token ids) and a host-side capacity ``cap`` >= count: the token-wise layers run on [cap, d] tensors (csrc/rows.cu)."""

    def __init__(self, tok: torch.Tensor, cap: int, keep_ids: bool = False):
        lib = L.load()
        L.require_cuda(tok)
        self.tok = tok.reshape(-1).contiguous()
        self.n = self.tok.numel()
        self.cap = int(cap)
        dev = tok.device
        self.rows = torch.empty(self.n, device=dev, dtype=torch.int32)
        # ids[r] = tok[rows[r]] (zeros past the count when the caller wants to use them as scatter keys)
        self._tgt = (torch.zeros if keep_ids else torch.empty)(max(self.n, self.cap), device=dev, dtype=torch.int64)
        self.ids = self._tgt[: self.cap]
        self.count = torch.empty(1, device=dev, dtype=torch.int32)
        nb = lib.rbm_compact_ws_bytes(self.n)
        ws = _ws("compact", nb, dev)
        check(lib.rbm_compact_labels(ptr(self.tok), self.n, ptr(self.rows), ptr(self._tgt), ptr(self.count), ptr(ws), nb, stream()),
              "compact_labels")
        count_launches(3)
        self.seq_start = None
        if tok.dim() == 2:  # first compact row of every sequence (the compact attention walks a sequence's rows)
            Bsz, Ln = tok.shape
            self.seq_start = torch.empty(Bsz + 1, device=dev, dtype=torch.int32)
            check(lib.rbm_rows_seq_start(ptr(self.rows), ptr(self.count), Bsz, Ln, ptr(self.seq_start), stream()), "rows_seq_start")
            count_launches()


def _rows_gather(x2, live, coef=None):
    lib = L.load()
    out = torch.empty(live.cap, x2.shape[1], device=x2.device, dtype=torch.float32)
    check(lib.rbm_rows_gather(ptr(x2), x2.stride(0), ptr(live.rows), ptr(live.count), live.cap, x2.shape[1], ptr(coef), ptr(out), stream()),
          "rows_gather")
    count_launches()
    return out


def _rows_scatter(xc, live, fill):
    lib = L.load()
    d = xc.shape[1]
    out = torch.empty(live.n, d, device=xc.device, dtype=torch.float32)
    check(lib.rbm_rows_scatter(ptr(xc), ptr(live.rows), ptr(live.count), live.cap, d, ptr(fill), ptr(live.tok), live.n, ptr(out), d, stream()),
          "rows_scatter")
    count_launches()
    return out


class RowsGatherFn(torch.autograd.Function):
    """[n, d] -> [cap, d]: the live rows in ascending order, zero rows after them."""

    @staticmethod
    def forward(ctx, x, live):
        x2 = _rows2d(x)
        ctx.live, ctx.shape = live, x.shape
        return _rows_gather(x2, live)

    @staticmethod
    def backward(ctx, dy):
        return _rows_scatter(dy.contiguous(), ctx.live, None).view(ctx.shape), None


class RowsScatterFn(torch.autograd.Function):
    """[cap, d] -> [n, d]: live rows back in place; the rows of padding positions hold ``fill`` ([d]; None = zeros)."""

    @staticmethod
    def forward(ctx, xc, fill, live):
        ctx.live, ctx.has_fill = live, fill is not None
        return _rows_scatter(xc.contiguous(), live, fill.contiguous() if fill is not None else None)

    @staticmethod
    def backward(ctx, dy):
        lib = L.load()
        live = ctx.live
        dy2 = _rows2d(dy)
        dxc = _rows_gather(dy2, live)
        dfill = None
        if ctx.has_fill and ctx.needs_input_grad[1]:
            d = dy2.shape[1]
            dfill = torch.empty(d, device=dy.device, dtype=torch.float32)
            nb = lib.rbm_rows_dead_colsum_ws_bytes(d)
            ws = _ws("rows_colsum", nb, dy.device)
            check(lib.rbm_rows_dead_colsum(ptr(dy2), dy2.stride(0), ptr(live.tok), live.n, d, ptr(dfill), ptr(ws), nb, stream()),
                  "rows_dead_colsum")
            count_launches(2)
        return dxc, dfill, None


def rows_gather(x, live):
    return RowsGatherFn.apply(x, live)


def rows_scatter(xc, fill, live):
    return RowsScatterFn.apply(xc, fill, live)


# --------------------------------------------------------------------------------------------- embedding
class EmbedFn(torch.autograd.Function):
    """out = keep * dropout(table[tok]*scale + pos)   (K1-K3, K12)."""

    @staticmethod
    def forward(ctx, tok, table, pos, scale, zero_pad, p, seed, site):
        lib = L.load()
        L.require_cuda(tok, table, pos)
        Bsz, Ln = tok.shape
        d = table.shape[1]
        if pos.shape[0] < Ln:
            raise RuntimeError("positional table has %d rows < sequence length %d" % (pos.shape[0], Ln))
        tok = tok.contiguous()
        out = torch.empty(Bsz, Ln, d, device=table.device, dtype=torch.float32)
        check(lib.rbm_embed_fwd(ptr(tok), ptr(table), ptr(pos), ptr(out), Bsz * Ln, Ln, d, table.shape[0], float(scale),
                                int(zero_pad), float(p), seed, site, stream()), "embed_fwd")
        count_launches()
        ctx.save_for_backward(tok)
        ctx.meta = (table.shape, pos.shape, float(scale), int(zero_pad), float(p), seed, site)
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = L.load()
        (tok,) = ctx.saved_tensors
        tshape, pshape, scale, zero_pad, p, seed, site = ctx.meta
        Bsz, Ln = tok.shape
        d = tshape[1]
        dout = dout.contiguous()
        g = torch.empty_like(dout)
        dpos = torch.zeros(pshape, device=dout.device, dtype=torch.float32)
        check(lib.rbm_embed_bwd(ptr(tok), ptr(dout), ptr(g), ptr(dpos), Bsz * Ln, Ln, d, zero_pad, p, seed, site, stream()),
              "embed_bwd")
        count_launches()
        dtable = torch.zeros(tshape, device=dout.device, dtype=torch.float32)
        scatter_add_sorted_(dtable, tok, g, None, scale, padding_idx=0)
        return None, dtable, dpos, None, None, None, None, None


class EmbedLiveFn(torch.autograd.Function):
    """The embedding stage (zero_pad = 1) handing out the live rows only: [cap, d] = rows_gather(EmbedFn(...)).  Backward never
    builds the [B, L, d] gradient: dropout mask, positional-table gradient and the table scatter run on the cap compact rows."""

    @staticmethod
    def forward(ctx, tok, table, pos, live, scale, p, seed, site):
        lib = L.load()
        L.require_cuda(tok, table, pos)
        Bsz, Ln = tok.shape
        d = table.shape[1]
        if pos.shape[0] < Ln:
            raise RuntimeError("positional table has %d rows < sequence length %d" % (pos.shape[0], Ln))
        tok = tok.contiguous()
        full = torch.empty(Bsz * Ln, d, device=table.device, dtype=torch.float32)
        check(lib.rbm_embed_fwd(ptr(tok), ptr(table), ptr(pos), ptr(full), Bsz * Ln, Ln, d, table.shape[0], float(scale), 1, float(p), seed,
                                site, stream()), "embed_fwd")
        count_launches()
        ctx.save_for_backward(tok)
        ctx.live, ctx.meta = live, (table.shape, pos.shape, float(scale), float(p), seed, site)
        return _rows_gather(full, live)

    @staticmethod
    def backward(ctx, dout):
        lib = L.load()
        (tok,) = ctx.saved_tensors
        live = ctx.live
        tshape, pshape, scale, p, seed, site = ctx.meta
        Bsz, Ln = tok.shape
        d = tshape[1]
        dout = dout.contiguous()
        g = torch.empty_like(dout)
        idx = torch.empty(live.cap, device=dout.device, dtype=torch.int64)
        dpos = torch.zeros(pshape, device=dout.device, dtype=torch.float32)
        nb = lib.rbm_embed_bwd_rows_ws_bytes(Ln, d)
        ws = _ws("embed_rows", nb, dout.device)
        check(lib.rbm_embed_bwd_rows(ptr(tok), ptr(live.rows), ptr(live.count), live.cap, ptr(dout), ptr(g), ptr(idx), ptr(dpos), Ln, d, p,
                                     seed, site, ptr(ws), nb, stream()), "embed_bwd_rows")
        count_launches(3)
        dtable = torch.zeros(tshape, device=dout.device, dtype=torch.float32)
        scatter_add_sorted_(dtable, idx, g, None, scale, padding_idx=0)
        return None, dtable, dpos, None, None, None, None, None


def embed_live_supported(Ln: int, d: int) -> bool:
    return Ln * d * 4 <= 96 * 1024


# --------------------------------------------------------------------------------------------- layernorm
class LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, gamma, beta, eps, flavour):
        lib = L.load()
        L.require_cuda(x, gamma, beta)
        x2 = _rows2d(x).contiguous()
        rows, d = x2.shape
        y = torch.empty_like(x2)
        stats = torch.empty(rows, 2, device=x.device, dtype=torch.float32)
        check(lib.rbm_layernorm_fwd(ptr(x2), ptr(gamma), ptr(beta), ptr(y), ptr(stats), rows, d, float(eps), int(flavour),
                                    stream()), "layernorm_fwd")
        count_launches()
        ctx.save_for_backward(x2, gamma, stats)
        ctx.meta = (float(eps), int(flavour), x.shape)
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        lib = L.load()
        x2, gamma, stats = ctx.saved_tensors
        eps, flavour, shape = ctx.meta
        rows, d = x2.shape
        dy2 = dy.reshape(rows, d).contiguous()
        dx = torch.empty_like(x2)
        dgamma = torch.empty_like(gamma)
        dbeta = torch.empty_like(gamma)
        nb = lib.rbm_layernorm_ws_bytes(rows, d)
        ws = _ws("ln", nb, x2.device)
        check(lib.rbm_layernorm_bwd(ptr(x2), ptr(gamma), ptr(dy2), ptr(stats), ptr(dx), ptr(dgamma), ptr(dbeta), rows, d, eps,
                                    flavour, ptr(ws), nb, stream()), "layernorm_bwd")
        count_launches(2)
        return dx.view(shape), dgamma, dbeta, None, None


def layernorm(x, gamma, beta, eps, flavour):
    return LayerNormFn.apply(x, gamma, beta, eps, flavour)


class LayerNormResidualFn(torch.autograd.Function):
    """(LN(x), x) for the pre-norm sublayer x + f(LN(x)) (NN/models/bert_modules/utils/sublayer.py:16-18): the second output
    is x itself, to be used as the residual operand, so that in backward the gradient arriving through the residual branch
    is added inside the LayerNorm-backward pass that writes dx (one launch less and one read/write of [B*L, d] less than
    autograd's separate accumulation)."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, flavour):
        lib = L.load()
        L.require_cuda(x, gamma, beta)
        x2 = _rows2d(x).contiguous()
        rows, d = x2.shape
        y = torch.empty_like(x2)
        stats = torch.empty(rows, 2, device=x.device, dtype=torch.float32)
        check(lib.rbm_layernorm_fwd(ptr(x2), ptr(gamma), ptr(beta), ptr(y), ptr(stats), rows, d, float(eps), int(flavour),
                                    stream()), "layernorm_fwd")
        count_launches()
        ctx.save_for_backward(x2, gamma, stats)
        ctx.meta = (float(eps), int(flavour), x.shape)
        return y.view(x.shape), x.view_as(x)

    @staticmethod
    def backward(ctx, dy, dres):
        lib = L.load()
        x2, gamma, stats = ctx.saved_tensors
        eps, flavour, shape = ctx.meta
        rows, d = x2.shape
        if dy is None:
            dy = torch.zeros(shape, device=x2.device, dtype=x2.dtype)
        dy2 = dy.reshape(rows, d).contiguous()
        dres2 = None if dres is None else dres.reshape(rows, d).contiguous()
        dx = torch.empty_like(x2)
        dgamma = torch.empty_like(gamma)
        dbeta = torch.empty_like(gamma)
        nb = lib.rbm_layernorm_ws_bytes(rows, d)
        ws = _ws("ln", nb, x2.device)
        check(lib.rbm_layernorm_bwd_residual(ptr(x2), ptr(gamma), ptr(dy2), ptr(dres2) if dres2 is not None else None, ptr(stats),
                                             ptr(dx), ptr(dgamma), ptr(dbeta), rows, d, eps, flavour, ptr(ws), nb, stream()),
              "layernorm_bwd_residual")
        count_launches(2)
        return dx.view(shape), dgamma, dbeta, None, None


class LayerNormFanoutFn(torch.autograd.Function):
    """(LN(x), LN(x), x): the normalised output for TWO consumers plus the input for a second consumer (SASRec block,
    NN/models/sas_model/sas.py:72-84: Q feeds the q-projection and the residual, x feeds LN and the k/v projection).  All three
    gradients meet inside one LayerNorm-backward launch (rbm_layernorm_bwd_fanout) instead of autograd's elementwise adds."""

    @staticmethod
    def forward(ctx, x, gamma, beta, eps, flavour):
        lib = L.load()
        L.require_cuda(x, gamma, beta)
        x2 = _rows2d(x).contiguous()
        rows, d = x2.shape
        y = torch.empty_like(x2)
        stats = torch.empty(rows, 2, device=x.device, dtype=torch.float32)
        check(lib.rbm_layernorm_fwd(ptr(x2), ptr(gamma), ptr(beta), ptr(y), ptr(stats), rows, d, float(eps), int(flavour),
                                    stream()), "layernorm_fwd")
        count_launches()
        ctx.save_for_backward(x2, gamma, stats)
        ctx.meta = (float(eps), int(flavour), x.shape)
        return y.view(x.shape), y.view(x.shape), x.view_as(x)

    @staticmethod
    def backward(ctx, dy, dy2, dres):
        lib = L.load()
        x2, gamma, stats = ctx.saved_tensors
        eps, flavour, shape = ctx.meta
        rows, d = x2.shape
        if dy is None:
            dy, dy2 = dy2, None
        if dy is None:
            dy = torch.zeros(shape, device=x2.device, dtype=x2.dtype)
        c2 = lambda t: None if t is None else t.reshape(rows, d).contiguous()
        dy, dy2, dres = c2(dy), c2(dy2), c2(dres)
        dx = torch.empty_like(x2)
        dgamma = torch.empty_like(gamma)
        dbeta = torch.empty_like(gamma)
        nb = lib.rbm_layernorm_ws_bytes(rows, d)
        ws = _ws("ln", nb, x2.device)
        check(lib.rbm_layernorm_bwd_fanout(ptr(x2), ptr(gamma), ptr(dy), ptr(dy2), ptr(dres), ptr(stats), ptr(dx), ptr(dgamma),
                                           ptr(dbeta), rows, d, eps, flavour, ptr(ws), nb, stream()), "layernorm_bwd_fanout")
        count_launches(2)
        return dx.view(shape), dgamma, dbeta, None, None


def layernorm_fanout(x, gamma, beta, eps, flavour):
    """-> (LN(x), LN(x) again for a second consumer, x for a second consumer); see LayerNormFanoutFn."""
    return LayerNormFanoutFn.apply(x, gamma, beta, eps, flavour)


def layernorm_residual(x, gamma, beta, eps, flavour):
    """-> (LN(x), x): use the second value as the residual operand of the sublayer (see LayerNormResidualFn)."""
    return LayerNormResidualFn.apply(x, gamma, beta, eps, flavour)


# ------------------------------------------------------------------------------------------------ linear
class LinearFn(torch.autograd.Function):
    """y = rowkeep * dropB(residual + dropA(act(x.w^T + b)))   (K6, K9-K12)."""

    @staticmethod
    def forward(ctx, x, w, bias, residual, row_tok, act, pA, siteA, pB, siteB, seed):
        lib = L.load()
        L.require_cuda(x, w)
        x2 = _rows2d(x)
        M, K = x2.shape
        N = w.shape[0]
        w = w.contiguous()
        y = torch.empty(M, N, device=x.device, dtype=torch.float32)
        need_pre = act != L.ACT_NONE and (x.requires_grad or w.requires_grad)
        pre = torch.empty(M, N, device=x.device, dtype=torch.float32) if need_pre else None
        res2 = _rows2d(residual) if residual is not None else None
        if row_tok is not None:
            row_tok = row_tok.reshape(-1).contiguous()
        nbf = lib.rbm_linear_fwd_ws_bytes(M, N, K)
        wsf = _ws("lin_fwd", nbf, x.device) if nbf else None
        check(lib.rbm_linear_fwd_ws(ptr(x2), x2.stride(0), ptr(w), ptr(bias), ptr(y), N, ptr(pre), M, N, K, int(act), ptr(res2),
                                    res2.stride(0) if res2 is not None else 0, ptr(row_tok), float(pA), siteA, float(pB), siteB,
                                    seed, ptr(wsf), nbf, stream()), "linear_fwd")
        count_launches(6 if nbf else 1)
        ctx.save_for_backward(x2, w, pre, row_tok)
        ctx.meta = (int(act), float(pA), siteA, float(pB), siteB, seed, bias is not None, residual is not None, x.shape,
                    residual.shape if residual is not None else None)
        return y.view(*x.shape[:-1], N)

    @staticmethod
    def backward(ctx, dy):
        lib = L.load()
        x2, w, pre, row_tok = ctx.saved_tensors
        act, pA, siteA, pB, siteB, seed, has_bias, has_res, xshape, rshape = ctx.meta
        M, K = x2.shape
        N = w.shape[0]
        dy2 = dy.reshape(M, N).contiguous()
        trivial = act == L.ACT_NONE and pA == 0.0 and pB == 0.0 and row_tok is None
        if trivial:
            dpre, dres = dy2, (dy2 if has_res else None)
        else:
            dpre = torch.empty_like(dy2)
            # dres is needed as a separate tensor only when something sits between the residual add and the output
            need_dres = has_res
            dres = torch.empty_like(dy2) if need_dres else None
            check(lib.rbm_linear_epilogue_bwd(ptr(dy2), ptr(pre), ptr(dpre), ptr(dres), M, N, act, ptr(row_tok), pA, siteA, pB,
                                              siteB, seed, stream()), "linear_epilogue_bwd")
            count_launches()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty(M, K, device=dy.device, dtype=torch.float32)
            nbd = lib.rbm_linear_bwd_data_ws_bytes(N, K)
            wsd = _ws("lin_dx", nbd, dy.device)
            check(lib.rbm_linear_bwd_data(ptr(dpre), N, ptr(w), ptr(dx), K, M, N, K, ptr(wsd), nbd, stream()), "linear_bwd_data")
            count_launches(2)
            dx = dx.view(xshape)
        if ctx.needs_input_grad[1] or (has_bias and ctx.needs_input_grad[2]):
            dw = torch.empty_like(w)
            db = torch.empty(N, device=dy.device, dtype=torch.float32) if has_bias else None
            nb = lib.rbm_linear_bwd_weight_ws_bytes(M, N, K)
            ws = _ws("lin_dw", nb, dy.device)
            check(lib.rbm_linear_bwd_weight(ptr(dpre), N, ptr(x2), x2.stride(0), ptr(dw), ptr(db), M, N, K, ptr(ws), nb, stream()),
                  "linear_bwd_weight")
            count_launches(2)  # partial dW (+ fused db) and the fixed-order reduction
        return dx, dw, db, (dres.view(rshape) if has_res else None), None, None, None, None, None, None, None


def linear(x, w, bias=None, residual=None, row_tok=None, act=L.ACT_NONE, pA=0.0, siteA=0, pB=0.0, siteB=0, seed=0):
    return LinearFn.apply(x, w, bias, residual, row_tok, act, pA, siteA, pB, siteB, seed)


# --------------------------------------------------------------------------------------------- attention
class AttnFn(torch.autograd.Function):
    """ctx = dropout(softmax(mask(scale q.k^T))).v, heads laid out as column blocks (K7-K9).

    ``a`` holds q (columns [qc, qc+d)); ``b`` (or ``a`` when b is None) holds k and v at columns kc / vc."""

    @staticmethod
    def forward(ctx, a, b, tok, Bsz, Ln, h, qc, kc, vc, mask_mode, scale, p, seed, site):
        lib = L.load()
        L.require_cuda(a, b)
        a2 = _rows2d(a)
        b2 = _rows2d(b) if b is not None else a2
        M = a2.shape[0]
        d = (a2.shape[1] // 3) if b is None else a2.shape[1]
        dk = d // h
        if tok is not None:
            tok = tok.reshape(-1).contiguous()
        out = torch.empty(M, d, device=a.device, dtype=torch.float32)
        stats = torch.empty(Bsz * h * Ln, 2, device=a.device, dtype=torch.float32)
        check(lib.rbm_attn_fwd(a2.data_ptr() + 4 * qc, a2.stride(0), b2.data_ptr() + 4 * kc, b2.stride(0), b2.data_ptr() + 4 * vc,
                               b2.stride(0), ptr(tok), ptr(out), d, ptr(stats), Bsz, Ln, h, dk, int(mask_mode), float(scale),
                               float(p), seed, site, stream()), "attn_fwd")
        count_launches()
        ctx.save_for_backward(a2, b2 if b is not None else None, tok, out, stats)
        ctx.meta = (Bsz, Ln, h, dk, d, qc, kc, vc, int(mask_mode), float(scale), float(p), seed, site, a.shape,
                    b.shape if b is not None else None)
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = L.load()
        a2, b2s, tok, out, stats = ctx.saved_tensors
        Bsz, Ln, h, dk, d, qc, kc, vc, mask_mode, scale, p, seed, site, ashape, bshape = ctx.meta
        b2 = b2s if b2s is not None else a2
        dout = dout.reshape(-1, d).contiguous()
        da = torch.empty_like(a2) if a2.is_contiguous() else torch.empty(a2.shape, device=a2.device, dtype=torch.float32)
        db = da if b2s is None else torch.empty(b2.shape, device=a2.device, dtype=torch.float32)
        nb = lib.rbm_attn_bwd_ws_bytes(Bsz, Ln, h)
        ws = _ws("attn", nb, a2.device)
        check(lib.rbm_attn_bwd(a2.data_ptr() + 4 * qc, a2.stride(0), b2.data_ptr() + 4 * kc, b2.stride(0),
                               b2.data_ptr() + 4 * vc, b2.stride(0), ptr(tok), ptr(out), d, ptr(dout), d, ptr(stats),
                               da.data_ptr() + 4 * qc, da.stride(0), db.data_ptr() + 4 * kc, db.stride(0),
                               db.data_ptr() + 4 * vc, db.stride(0), Bsz, Ln, h, dk, mask_mode, scale, p, seed, site, ptr(ws),
                               nb, stream()), "attn_bwd")
        count_launches(2)
        return (da.view(ashape), (db.view(bshape) if b2s is not None else None)) + (None,) * 12


def attention(a, b, tok, Bsz, Ln, h, qc, kc, vc, mask_mode, scale, p=0.0, seed=0, site=0):
    return AttnFn.apply(a, b, tok, Bsz, Ln, h, qc, kc, vc, mask_mode, scale, p, seed, site)


class AttnLqFn(torch.autograd.Function):
    """Attention with per-sequence compacted queries: ``q`` [B*Lq, d] (Lq rows per sequence, zero rows after the real ones) against
    the keys / values of all L positions, ``kv`` [B*L, 2d] (k | v).  Tensor path only (rbm_attn_fwd_lq / rbm_attn_bwd_lq)."""

    @staticmethod
    def forward(ctx, q, kv, tok, Bsz, Ln, Lq, h, mask_mode, scale, p, seed, site):
        lib = L.load()
        L.require_cuda(q, kv)
        q, kv = q.contiguous(), kv.contiguous()
        d = q.shape[1]
        if tok is not None:
            tok = tok.reshape(-1).contiguous()
        out = torch.empty(Bsz * Lq, d, device=q.device, dtype=torch.float32)
        stats = torch.empty(Bsz * h * Lq, 2, device=q.device, dtype=torch.float32)
        check(lib.rbm_attn_fwd_lq(ptr(q), d, ptr(kv), 2 * d, kv.data_ptr() + 4 * d, 2 * d, ptr(tok), ptr(out), d, ptr(stats), Bsz, Ln, Lq,
                                  h, d // h, int(mask_mode), float(scale), float(p), seed, site, stream()), "attn_fwd_lq")
        count_launches()
        ctx.save_for_backward(q, kv, tok, out, stats)
        ctx.meta = (Bsz, Ln, Lq, h, d, int(mask_mode), float(scale), float(p), seed, site)
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = L.load()
        q, kv, tok, out, stats = ctx.saved_tensors
        Bsz, Ln, Lq, h, d, mask_mode, scale, p, seed, site = ctx.meta
        dout = dout.contiguous()
        dq = torch.empty_like(q)
        dkv = torch.empty_like(kv)
        nb = lib.rbm_attn_bwd_lq_ws_bytes(Bsz, Lq, h)
        ws = _ws("attn", nb, q.device)
        check(lib.rbm_attn_bwd_lq(ptr(q), d, ptr(kv), 2 * d, kv.data_ptr() + 4 * d, 2 * d, ptr(tok), ptr(out), d, ptr(dout), d, ptr(stats),
                                  ptr(dq), d, ptr(dkv), 2 * d, dkv.data_ptr() + 4 * d, 2 * d, Bsz, Ln, Lq, h, d // h, mask_mode, scale, p,
                                  seed, site, ptr(ws), nb, stream()), "attn_bwd_lq")
        count_launches(2)
        return (dq, dkv) + (None,) * 10


def attention_lq(q, kv, tok, Bsz, Ln, Lq, h, mask_mode, scale, p=0.0, seed=0, site=0):
    return AttnLqFn.apply(q, kv, tok, Bsz, Ln, Lq, h, mask_mode, scale, p, seed, site)


def attention_lq_supported(Ln, Lq, dk, mask_mode) -> bool:
    return bool(L.load().rbm_attn_lq_supported(int(Ln), int(Lq), int(dk), int(mask_mode)))


def _rows_to_seq(xc, live, Bsz, Lq):
    lib = L.load()
    d = xc.shape[1]
    out = torch.empty(Bsz * Lq, d, device=xc.device, dtype=torch.float32)
    check(lib.rbm_rows_to_seq(ptr(xc), ptr(live.seq_start), Bsz, Lq, d, ptr(out), stream()), "rows_to_seq")
    count_launches()
    return out


def _seq_to_rows(xs, live, Ln, Lq):
    lib = L.load()
    d = xs.shape[1]
    out = torch.empty(live.cap, d, device=xs.device, dtype=torch.float32)
    check(lib.rbm_seq_to_rows(ptr(xs), ptr(live.rows), ptr(live.seq_start), ptr(live.count), live.cap, Ln, Lq, d, ptr(out), stream()),
          "seq_to_rows")
    count_launches()
    return out


class RowsToSeqFn(torch.autograd.Function):
    """[cap, d] compact rows -> [B*Lq, d]: slot o of sequence b = its o-th live row, zero rows after the last one."""

    @staticmethod
    def forward(ctx, xc, live, Bsz, Ln, Lq):
        ctx.live, ctx.meta = live, (Bsz, Ln, Lq)
        return _rows_to_seq(xc.contiguous(), live, Bsz, Lq)

    @staticmethod
    def backward(ctx, dy):
        Bsz, Ln, Lq = ctx.meta
        return _seq_to_rows(dy.contiguous(), ctx.live, Ln, Lq), None, None, None, None


class SeqToRowsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, xs, live, Bsz, Ln, Lq):
        ctx.live, ctx.meta = live, (Bsz, Ln, Lq)
        return _seq_to_rows(xs.contiguous(), live, Ln, Lq)

    @staticmethod
    def backward(ctx, dy):
        Bsz, Ln, Lq = ctx.meta
        return _rows_to_seq(dy.contiguous(), ctx.live, Bsz, Lq), None, None, None, None


def rows_to_seq(xc, live, Bsz, Ln, Lq):
    return RowsToSeqFn.apply(xc, live, Bsz, Ln, Lq)


def seq_to_rows(xs, live, Bsz, Ln, Lq):
    return SeqToRowsFn.apply(xs, live, Bsz, Ln, Lq)


class AttnLiveFn(torch.autograd.Function):
    """SASRec causal attention on the compact live-row layout (csrc/attention_live.cu): q [cap, d], kv [cap, 2d] (k | v), every
    padding position's key / value = bkv [2d].  Rows past the live count stay zero."""

    @staticmethod
    def forward(ctx, q, kv, bkv, live, Bsz, Ln, h, scale, p, seed, site):
        lib = L.load()
        L.require_cuda(q, kv, bkv)
        q, kv, bkv = q.contiguous(), kv.contiguous(), bkv.contiguous()
        cap, d = q.shape
        out = torch.zeros(cap, d, device=q.device, dtype=torch.float32)
        stats = torch.empty(cap, h, 2, device=q.device, dtype=torch.float32)
        check(lib.rbm_attn_live_fwd(ptr(q), d, ptr(kv), 2 * d, ptr(bkv), ptr(live.rows), ptr(live.seq_start), ptr(live.tok), ptr(out),
                                    ptr(stats), Bsz, Ln, h, d // h, float(scale), float(p), seed, site, stream()), "attn_live_fwd")
        count_launches(2)
        ctx.save_for_backward(q, kv, bkv, out, stats)
        ctx.live, ctx.meta = live, (Bsz, Ln, h, float(scale), float(p), seed, site)
        return out

    @staticmethod
    def backward(ctx, dout):
        lib = L.load()
        q, kv, bkv, out, stats = ctx.saved_tensors
        live = ctx.live
        Bsz, Ln, h, scale, p, seed, site = ctx.meta
        cap, d = q.shape
        dout = dout.contiguous()
        dq = torch.zeros_like(q)
        dkv = torch.zeros_like(kv)
        dead = torch.zeros_like(kv)
        delta = torch.empty(cap, h, device=q.device, dtype=torch.float32)
        keepw = torch.empty(cap, h, device=q.device, dtype=torch.int64)
        check(lib.rbm_attn_live_bwd(ptr(q), d, ptr(kv), 2 * d, ptr(bkv), ptr(live.rows), ptr(live.seq_start), ptr(live.tok), ptr(out),
                                    ptr(stats), ptr(dout), ptr(dq), ptr(dkv), ptr(dead), ptr(delta), ptr(keepw), Bsz, Ln, h, d // h, scale,
                                    p, seed, site, stream()), "attn_live_bwd")
        dbkv = torch.empty(2 * d, device=q.device, dtype=torch.float32)
        nb = lib.rbm_rows_dead_colsum_ws_bytes(2 * d)
        ws = _ws("rows_colsum", nb, q.device)
        check(lib.rbm_rows_live_colsum(ptr(dead), 2 * d, ptr(live.count), cap, 2 * d, ptr(dbkv), ptr(ws), nb, stream()), "rows_live_colsum")
        count_launches(7)
        return dq, dkv, dbkv, None, None, None, None, None, None, None, None


def attention_live(q, kv, bkv, live, Bsz, Ln, h, scale, p=0.0, seed=0, site=0):
    return AttnLiveFn.apply(q, kv, bkv, live, Bsz, Ln, h, scale, p, seed, site)


def attention_last_query(q, kv, tok, Bsz, Ln, h, kc, vc, mask_mode, scale):
    """Evaluation only (K20): context of the last position of every sequence.  ``q`` [B, h*dk] holds the last position's query,
    ``kv`` [B*L, cols] the keys (columns [kc, kc+d)) and values ([vc, vc+d)) of every position.  No autograd, no dropout."""
    lib = L.load()
    L.require_cuda(q, kv)
    if torch.is_grad_enabled() and (q.requires_grad or kv.requires_grad):
        raise RuntimeError("attention_last_query is an evaluation-only op (no backward): call it under torch.no_grad()")
    q2, kv2 = _rows2d(q), _rows2d(kv)
    d = q2.shape[1]
    out = torch.empty(Bsz, d, device=q.device, dtype=torch.float32)
    if tok is not None:
        tok = tok.reshape(-1).contiguous()
    check(lib.rbm_attn_last_query(ptr(q2), q2.stride(0), kv2.data_ptr() + 4 * kc, kv2.stride(0), kv2.data_ptr() + 4 * vc, kv2.stride(0),
                                  ptr(tok), ptr(out), d, Bsz, Ln, h, d // h, int(mask_mode), float(scale), stream()), "attn_last_query")
    count_launches()
    return out


# ---------------------------------------------------------------------- BERT scoring + masked cross-entropy
class ScoreCEFn(torch.autograd.Function):
    """loss = mean over labels != 0 of (logsumexp(h.w^T + b) - target logit); logits never materialised (K15-K16)."""

    @staticmethod
    def forward(ctx, hidden, labels, w, bias):
        lib = L.load()
        L.require_cuda(hidden, labels, w, bias)
        h2 = _rows2d(hidden).contiguous()
        n, d = h2.shape
        V1 = w.shape[0]
        labels = labels.reshape(-1).contiguous()
        dev = hidden.device
        rows = torch.empty(n, device=dev, dtype=torch.int32)
        tgt = torch.empty(n, device=dev, dtype=torch.int64)
        count = torch.empty(1, device=dev, dtype=torch.int32)
        nb = lib.rbm_compact_ws_bytes(n)
        ws = _ws("compact", nb, dev)
        check(lib.rbm_compact_labels(ptr(labels), n, ptr(rows), ptr(tgt), ptr(count), ptr(ws), nb, stream()), "compact_labels")
        lse = torch.empty(n, device=dev, dtype=torch.float32)
        loss = torch.empty((), device=dev, dtype=torch.float32)
        nb = lib.rbm_ce_ws_bytes(n, V1, d)
        ws = _ws("ce", nb, dev)
        w = w.contiguous()
        check(lib.rbm_ce_fwd(ptr(h2), ptr(rows), ptr(tgt), ptr(count), ptr(w), ptr(bias), ptr(lse), ptr(loss), n, V1, d, ptr(ws),
                             nb, stream()), "ce_fwd")
        count_launches(5)
        ctx.save_for_backward(h2, rows, tgt, count, w, bias, lse)
        ctx.shape = hidden.shape
        return loss

    @staticmethod
    def backward(ctx, dloss):
        lib = L.load()
        h2, rows, tgt, count, w, bias, lse = ctx.saved_tensors
        n, d = h2.shape
        V1 = w.shape[0]
        dloss = dloss.reshape(1).contiguous().float()
        dh = torch.zeros_like(h2)
        dw = torch.empty_like(w)
        db = torch.empty(V1, device=h2.device, dtype=torch.float32)
        nb = lib.rbm_ce_ws_bytes(n, V1, d)
        ws = _ws("ce", nb, h2.device)
        check(lib.rbm_ce_bwd(ptr(h2), ptr(rows), ptr(tgt), ptr(count), ptr(w), ptr(bias), ptr(lse), ptr(dloss), ptr(dh), ptr(dw),
                             ptr(db), n, V1, d, ptr(ws), nb, stream()), "ce_bwd")
        count_launches(4)
        return dh.view(ctx.shape), None, dw, db


def score_cross_entropy(hidden, labels, w, bias):
    return ScoreCEFn.apply(hidden, labels, w, bias)


# ------------------------------------------------------------------------------------ SASRec scoring + BCE
class SasScoreFn(torch.autograd.Function):
    """pos/neg logits = <f, table[pos]> / <f, table[neg]>   (K13)."""

    @staticmethod
    def forward(ctx, f, table, pos, neg, cap=None):
        lib = L.load()
        L.require_cuda(f, table, pos, neg)
        ctx.cap = cap
        f2 = _rows2d(f).contiguous()
        rows, d = f2.shape
        pos = pos.reshape(-1).contiguous()
        neg = neg.reshape(-1).contiguous()
        pl = torch.empty(rows, device=f.device, dtype=torch.float32)
        nl = torch.empty(rows, device=f.device, dtype=torch.float32)
        check(lib.rbm_sas_score_fwd(ptr(f2), ptr(table), ptr(pos), ptr(neg), ptr(pl), ptr(nl), rows, d, stream()), "sas_score_fwd")
        count_launches()
        ctx.save_for_backward(f2, table, pos, neg)
        ctx.shape = f.shape
        return pl.view(f.shape[:-1]), nl.view(f.shape[:-1])

    @staticmethod
    def backward(ctx, dpl, dnl):
        lib = L.load()
        f2, table, pos, neg = ctx.saved_tensors
        rows, d = f2.shape
        dpl = dpl.reshape(-1).contiguous()
        dnl = dnl.reshape(-1).contiguous()
        df = torch.empty_like(f2)
        check(lib.rbm_sas_score_bwd(ptr(table), ptr(pos), ptr(neg), ptr(dpl), ptr(dnl), ptr(df), rows, d, stream()), "sas_score_bwd")
        count_launches()
        dtable = torch.zeros_like(table)
        if ctx.cap is None:
            scatter_add_sorted_(dtable, pos, f2, dpl, 1.0, padding_idx=0)
            scatter_add_sorted_(dtable, neg, f2, dnl, 1.0, padding_idx=0)
        else:
            # at most `cap` ids are non-zero (the caller's promise, see SASModel._live_rows): sort and reduce those entries only
            # (same contributions, the coefficient folded in with the same rounding) ...
            # ... and both id lists in ONE sort / segment reduction: [positive entries ; negative entries], cap each
            cap = ctx.cap
            ids = torch.empty(2 * cap, device=f2.device, dtype=torch.int64)
            src = torch.empty(2 * cap, d, device=f2.device, dtype=torch.float32)
            for k, (idx, coef) in enumerate(((pos, dpl), (neg, dnl))):
                lr = LiveRows(idx, cap, keep_ids=True)
                ids[k * cap:(k + 1) * cap].copy_(lr.ids)
                check(lib.rbm_rows_gather(ptr(f2), f2.stride(0), ptr(lr.rows), ptr(lr.count), cap, d, ptr(coef),
                                          src.data_ptr() + 4 * k * cap * d, stream()), "rows_gather")
                count_launches(2)
            scatter_add_sorted_(dtable, ids, src, None, 1.0, padding_idx=0)
        return df.view(ctx.shape), dtable, None, None, None


def sas_scores(f, table, pos, neg, cap=None):
    """``cap``: an upper bound (rows) on the number of non-zero ids in ``pos`` and in ``neg``; the table gradient then sorts /
    reduces ``cap`` entries instead of B*L."""
    return SasScoreFn.apply(f, table, pos, neg, cap)


class BcePairFn(torch.autograd.Function):
    """mean_{pos!=0} BCEWithLogits(pl, 1) + mean_{pos!=0} BCEWithLogits(nl, 0)   (K14)."""

    @staticmethod
    def forward(ctx, pl, nl, pos):
        lib = L.load()
        L.require_cuda(pl, nl, pos)
        plc, nlc, posc = pl.reshape(-1).contiguous(), nl.reshape(-1).contiguous(), pos.reshape(-1).contiguous()
        rows = plc.numel()
        loss = torch.empty((), device=pl.device, dtype=torch.float32)
        count = torch.empty(1, device=pl.device, dtype=torch.int32)
        nb = lib.rbm_bce_ws_bytes(rows)
        ws = _ws("bce", nb, pl.device)
        check(lib.rbm_bce_pair_fwd(ptr(plc), ptr(nlc), ptr(posc), ptr(loss), ptr(count), rows, ptr(ws), nb, stream()), "bce_pair_fwd")
        count_launches(2)
        ctx.save_for_backward(plc, nlc, posc, count)
        ctx.shape = pl.shape
        return loss

    @staticmethod
    def backward(ctx, dloss):
        lib = L.load()
        plc, nlc, posc, count = ctx.saved_tensors
        dloss = dloss.reshape(1).contiguous().float()
        dpl = torch.empty_like(plc)
        dnl = torch.empty_like(nlc)
        check(lib.rbm_bce_pair_bwd(ptr(plc), ptr(nlc), ptr(posc), ptr(count), ptr(dloss), ptr(dpl), ptr(dnl), plc.numel(), stream()),
              "bce_pair_bwd")
        count_launches()
        return dpl.view(ctx.shape), dnl.view(ctx.shape), None


def bce_pair_loss(pl, nl, pos):
    return BcePairFn.apply(pl, nl, pos)


# ------------------------------------------------------------------------------------- evaluation kernels
def candidate_scores(f, table, bias, cand):
    """out[u,c] = <table[cand[u,c]], f[u]> (+bias)  -- sampled-candidate evaluation (K19 with C=101)."""
    lib = L.load()
    L.require_cuda(f, table, cand)
    f2 = _rows2d(f)
    cand = cand.contiguous()
    U, Cn = cand.shape
    out = torch.empty(U, Cn, device=f.device, dtype=torch.float32)
    check(lib.rbm_candidate_scores(ptr(f2), f2.stride(0), ptr(table), ptr(bias), ptr(cand), ptr(out), U, Cn, table.shape[1], stream()),
          "candidate_scores")
    count_launches()
    return out


def score_topk(f, table, bias, v_begin, v_end, k, id_offset=0, exclude=None):
    """Fused full-catalogue scoring + top-k over table rows [v_begin, v_end)  (K19-K21); ids = row + id_offset.

    ``exclude`` (optional ``[U, n]`` int64 CUDA tensor): row u lists ids (same id space as the result) that user u must not be
    ranked, in any order, with duplicates allowed; ids <= 0 are padding.  The result is then the top-k of the remaining items
    (trailing ``(-inf, -1)`` when fewer than k remain)."""
    lib = L.load()
    L.require_cuda(f, table)
    f2 = _rows2d(f)
    U, d = f2.shape
    ex, n_ex = None, 0
    if exclude is not None:
        if not torch.is_tensor(exclude) or not exclude.is_cuda or exclude.device != f.device:
            raise RuntimeError("score_topk: exclude must be a CUDA tensor on the device of f")
        if exclude.dtype != torch.int64 or exclude.dim() != 2 or exclude.shape[0] != U:
            raise RuntimeError("score_topk: exclude must be int64 [U=%d, n], got %s %s" % (U, exclude.dtype, tuple(exclude.shape)))
        n_ex = int(exclude.shape[1])
        if n_ex > 0:
            ex = exclude
            if v_begin + id_offset <= 0:  # ids <= 0 are real items of this call: keep the padding from matching them
                ex = ex.masked_fill(ex <= 0, torch.iinfo(torch.int64).min)
            ex = torch.sort(ex, dim=1).values.contiguous()  # the kernels walk each row in ascending order
    vals = torch.empty(U, k, device=f.device, dtype=torch.float32)
    ids = torch.empty(U, k, device=f.device, dtype=torch.int64)
    nb = lib.rbm_score_topk_ws_bytes_d(U, v_end - v_begin, d, k)
    ws = _ws("topk", nb, f.device)
    if ex is None:
        check(lib.rbm_score_topk(ptr(f2), f2.stride(0), ptr(table), ptr(bias), v_begin, v_end, id_offset, ptr(vals), ptr(ids), U, d, k,
                                 ptr(ws), nb, stream()), "score_topk")
    else:
        check(lib.rbm_score_topk_excl(ptr(f2), f2.stride(0), ptr(table), ptr(bias), v_begin, v_end, id_offset, ptr(ex), ex.stride(0), n_ex,
                                      ptr(vals), ptr(ids), U, d, k, ptr(ws), nb, stream()), "score_topk")
    count_launches(2)
    return vals, ids


def topk_rows(scores, k, id_offset=0):
    lib = L.load()
    L.require_cuda(scores)
    s2 = _rows2d(scores)
    U, Cn = s2.shape
    vals = torch.empty(U, k, device=scores.device, dtype=torch.float32)
    ids = torch.empty(U, k, device=scores.device, dtype=torch.int64)
    check(lib.rbm_topk_rows(ptr(s2), s2.stride(0), ptr(vals), ptr(ids), U, Cn, k, id_offset, stream()), "topk_rows")
    count_launches()
    return vals, ids


def topk_merge(vals, ids):
    """[S,U,k] per-shard lists -> [U,k]."""
    lib = L.load()
    L.require_cuda(vals, ids)
    S, U, k = vals.shape
    vals, ids = vals.contiguous(), ids.contiguous()
    ov = torch.empty(U, k, device=vals.device, dtype=torch.float32)
    oi = torch.empty(U, k, device=vals.device, dtype=torch.int64)
    check(lib.rbm_topk_merge(ptr(vals), ptr(ids), ptr(ov), ptr(oi), S, U, k, stream()), "topk_merge")
    count_launches()
    return ov, oi


_weight_cache = {}


def _rank_weights(K, device):
    """1/log2(t+2) and 1/(t+1) tables, computed by torch on the CPU exactly as NN/trainers/utils.py:43-44,51-52."""
    key = (K, str(device))
    if key not in _weight_cache:
        w_ndcg = 1 / torch.log2(torch.arange(2, 2 + K).float())
        w_mrr = 1 / torch.arange(1, K + 1).float()
        _weight_cache[key] = (w_ndcg.to(device), w_mrr.to(device))
    return _weight_cache[key]


def rank_metrics(top_ids, ks, labels=None, positives=None, id_offset=0):
    """per-user [U, len(ks), 3] = (Recall@k, NDCG@k, MRR@k)   (K22)."""
    lib = L.load()
    L.require_cuda(top_ids)
    U, K = top_ids.shape
    ks = [int(k) for k in ks]
    w_ndcg, w_mrr = _rank_weights(K, top_ids.device)
    per_user = torch.empty(U, len(ks), 3, device=top_ids.device, dtype=torch.float32)
    ks_arr = (C.c_int32 * len(ks))(*ks)
    Cn = labels.shape[1] if labels is not None else 0
    if labels is not None:
        labels = labels.contiguous()
    if positives is not None:
        positives = positives.contiguous()
    check(lib.rbm_rank_metrics(ptr(top_ids.contiguous()), ptr(labels), ptr(positives), ptr(w_ndcg), ptr(w_mrr),
                               C.cast(ks_arr, C.c_void_p), len(ks), ptr(per_user), U, K, Cn, id_offset, stream()), "rank_metrics")
    count_launches()
    return per_user


def column_mean(x):
    lib = L.load()
    L.require_cuda(x)
    x2 = x.reshape(x.shape[0], -1).contiguous()
    U, cols = x2.shape
    out = torch.empty(cols, device=x.device, dtype=torch.float32)
    nb = lib.rbm_column_mean_ws_bytes(U, cols)
    ws = _ws("colmean", nb, x.device)
    check(lib.rbm_column_mean(ptr(x2), ptr(out), U, cols, ptr(ws), nb, stream()), "column_mean")
    count_launches(2)
    return out


def dropout_mask(n, p, seed, site, device):
    """Debug/test: the keep mask an elementwise dropout site uses."""
    lib = L.load()
    out = torch.empty(n, device=device, dtype=torch.uint8)
    check(lib.rbm_dropout_mask(ptr(out), n, float(p), seed, site, stream()), "dropout_mask")
    return out


def dropout_mask_attn(rows, Ln, p, seed, site, device):
    lib = L.load()
    out = torch.empty(rows, Ln, device=device, dtype=torch.uint8)
    check(lib.rbm_dropout_mask_attn(ptr(out), rows, Ln, float(p), seed, site, stream()), "dropout_mask_attn")
    return out

# ------------------------------------------------------------------------------------ device-side batch construction
BATCH_SITE_BASE = 1 << 62  # Philox sites of batch construction live far away from the dropout sites (step*64 + local id)


def bert_cloze_batch(hist_ptr, hist_items, users, max_len, mask_prob, mask_token, num_items, seed, step):
    """(tokens, labels) int64 [B, L] on the device: Cloze masking of BertTrainDataset.__getitem__
    (NN/dataloaders/bert.py:77-110) from a CSR of user histories; a pure function of (histories, users, seed, step)."""
    lib = L.load()
    L.require_cuda(hist_ptr, hist_items, users)
    Bsz = int(users.numel())
    tokens = torch.empty(Bsz, max_len, device=users.device, dtype=torch.int64)
    labels = torch.empty(Bsz, max_len, device=users.device, dtype=torch.int64)
    check(lib.rbm_bert_cloze_batch(ptr(hist_ptr), ptr(hist_items), ptr(users), Bsz, int(max_len), float(mask_prob), int(mask_token),
                                   int(num_items), int(seed), BATCH_SITE_BASE + int(step), ptr(tokens), ptr(labels), stream()),
          "bert_cloze_batch")
    count_launches()
    return tokens, labels


def sas_train_batch(hist_ptr, hist_items, users, max_len, num_items, seed, step):
    """(seq, pos, neg) int64 [B, L] on the device: sample_function / random_neq of NN/dataloaders/sas.py:65-86."""
    lib = L.load()
    L.require_cuda(hist_ptr, hist_items, users)
    Bsz = int(users.numel())
    out = [torch.empty(Bsz, max_len, device=users.device, dtype=torch.int64) for _ in range(3)]
    check(lib.rbm_sas_train_batch(ptr(hist_ptr), ptr(hist_items), ptr(users), Bsz, int(max_len), int(num_items), int(seed),
                                  BATCH_SITE_BASE + int(step), ptr(out[0]), ptr(out[1]), ptr(out[2]), stream()), "sas_train_batch")
    count_launches()
    return tuple(out)


NEG_SITE = 1 << 41  # Philox site of the evaluation-negative sampler (disjoint from dropout and batch sites)


def negative_samples(seen_ptr, seen_items, num_items, n_samples, seed, pop_cdf=None, user_begin=0, num_users=None):
    """[num_users, n_samples] int64 evaluation negatives on the device: Random / PopularNegativeSampler
    (NN/dataloaders/negative_samplers/random.py:13-37, popular.py:15-44).  ``seen_items`` ascending + unique per user;
    ``pop_cdf`` (int64/uint64 [num_items], inclusive prefix sums of item counts) selects popularity-weighted draws."""
    lib = L.load()
    L.require_cuda(seen_ptr, seen_items)
    if pop_cdf is not None:
        L.require_cuda(pop_cdf)
        if pop_cdf.numel() != num_items or pop_cdf.dtype != torch.int64:
            raise RuntimeError("negative_samples: pop_cdf must be int64 [num_items]")
    U = int(seen_ptr.numel()) - 1 - int(user_begin) if num_users is None else int(num_users)
    out = torch.empty(U, int(n_samples), device=seen_ptr.device, dtype=torch.int64)
    check(lib.rbm_negative_samples(ptr(seen_ptr), ptr(seen_items), ptr(pop_cdf) if pop_cdf is not None else None, int(user_begin), U,
                                   int(num_items), int(n_samples), int(seed), NEG_SITE, ptr(out), stream()), "negative_samples")
    count_launches()
    return out


def eval_batch(hist_ptr, hist_items, answers, negatives, users, max_len, mask_token=-1):
    """(seq [B,L], candidates [B,1+N], labels [B,1+N]) int64 on the device: BertEvalDataset / SASEvalDataset.__getitem__
    (NN/dataloaders/bert.py:128-142 with ``mask_token`` appended, sas.py:136-153 with ``mask_token=-1``)."""
    lib = L.load()
    L.require_cuda(hist_ptr, hist_items, answers, users)
    Bsz = int(users.numel())
    n_neg = 0 if negatives is None else int(negatives.shape[1])
    if negatives is not None:
        L.require_cuda(negatives)
        negatives = negatives.contiguous()
    dev = users.device
    seq = torch.empty(Bsz, int(max_len), device=dev, dtype=torch.int64)
    cand = torch.empty(Bsz, 1 + n_neg, device=dev, dtype=torch.int64)
    labels = torch.empty(Bsz, 1 + n_neg, device=dev, dtype=torch.int64)
    check(lib.rbm_eval_batch(ptr(hist_ptr), ptr(hist_items), ptr(answers), ptr(negatives) if negatives is not None else None, ptr(users),
                             Bsz, int(max_len), n_neg, int(mask_token), ptr(seq), ptr(cand), ptr(labels), stream()), "eval_batch")
    count_launches()
    return seq, cand, labels
