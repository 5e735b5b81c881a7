"""Kernel-level parity: every C-ABI entry point vs the CPU oracle on seeded inputs (run with -m gpu on a B200)."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import rbm_b200
from rbm_b200 import ops, lib as L
from oracle import common as oc, metrics as om, optim as oo

pytestmark = pytest.mark.gpu
DEV = "cuda"


def g(x):
    return x.to(DEV)


def close(a, b, rtol=1e-4, atol=1e-5, msg=""):
    np.testing.assert_allclose(a.detach().cpu().numpy(), b.detach().cpu().numpy(), rtol=rtol, atol=atol, err_msg=msg)


# ------------------------------------------------------------------------------------------- embedding
@pytest.mark.parametrize("zero_pad,scale", [(1, 8.0), (0, 1.0)])
@pytest.mark.parametrize("p", [0.0, 0.25])
def test_embed_fwd_bwd(zero_pad, scale, p):
    torch.manual_seed(0)
    B, Ln, d, V = 5, 12, 32, 41
    tok = torch.randint(0, V, (B, Ln))
    tok[0, :4] = 0
    table = torch.randn(V, d)
    pos = torch.randn(Ln, d)
    dout = torch.randn(B, Ln, d)
    seed, site = 1234, 7
    tg, pg = g(table).requires_grad_(True), g(pos).requires_grad_(True)
    out = ops.EmbedFn.apply(g(tok), tg, pg, scale, zero_pad, p, seed, site)
    out.backward(g(dout))
    mask = ops.dropout_mask(B * Ln * d, p, seed, site, DEV).cpu().view(B, Ln, d) if p > 0 else None
    tr, pr = table.clone().requires_grad_(True), pos.clone().requires_grad_(True)
    ref = F.embedding(tok, tr, padding_idx=0) * scale + pr.unsqueeze(0)
    if p > 0:
        assert abs(mask.float().mean().item() - (1 - p)) < 0.03
        ref = ref * mask * (1.0 / (1.0 - p))
    if zero_pad:
        ref = ref * (tok != 0).unsqueeze(-1)
    ref.backward(dout)
    close(out, ref, 1e-6, 1e-6)
    close(pg.grad, pr.grad, 1e-5, 1e-5)
    close(tg.grad, tr.grad, 1e-5, 1e-5)


def test_embed_bad_shapes_raise():
    with pytest.raises(RuntimeError):
        ops.EmbedFn.apply(g(torch.zeros(2, 4, dtype=torch.long)), g(torch.randn(5, 6)), g(torch.randn(4, 6)), 1.0, 0, 0.0, 0, 0)
    with pytest.raises(RuntimeError):  # CPU tensors are refused: there is no fallback
        ops.EmbedFn.apply(torch.zeros(2, 4, dtype=torch.long), torch.randn(5, 8), torch.randn(4, 8), 1.0, 0, 0.0, 0, 0)


# ------------------------------------------------------------------------------------------ scatter-add
@pytest.mark.parametrize("n,V,d", [(400, 53, 16), (5000, 3418, 64), (70000, 12102, 128), (3, 300000, 8)])
def test_scatter_add_bit_exact(n, V, d):
    rng = np.random.RandomState(n)
    idx = (rng.zipf(1.2, size=n) % V).astype(np.int64)
    rows = rng.randn(n, d).astype(np.float32)
    coef = rng.randn(n).astype(np.float32)
    ref = oc.embedding_grad_scatter_chunked(idx, rows, V, padding_idx=0)
    short = np.bincount(idx, minlength=V) <= 64  # rows with <= 64 contributions: the reference's own order, bit for bit
    np.testing.assert_array_equal(ref[short], oc.embedding_grad_scatter_fast(idx, rows, V, padding_idx=0)[short])
    grad = torch.zeros(V, d, device=DEV)
    ops.scatter_add_sorted_(grad, g(torch.from_numpy(idx)), g(torch.from_numpy(rows)), None, 1.0, 0)
    np.testing.assert_array_equal(grad.cpu().numpy(), ref)  # bit-exact, run-to-run and vs the CPU order
    grad2 = torch.zeros(V, d, device=DEV)
    ops.scatter_add_sorted_(grad2, g(torch.from_numpy(idx)), g(torch.from_numpy(rows)), None, 1.0, 0)
    assert torch.equal(grad, grad2)
    ref_c = oc.embedding_grad_scatter_chunked(idx, rows * coef[:, None], V, padding_idx=0)
    grad3 = torch.zeros(V, d, device=DEV)
    ops.scatter_add_sorted_(grad3, g(torch.from_numpy(idx)), g(torch.from_numpy(rows)), g(torch.from_numpy(coef)), 1.0, 0)
    np.testing.assert_array_equal(grad3.cpu().numpy(), ref_c)
    assert grad.cpu()[0].abs().sum() == 0  # padding row untouched


def test_scatter_golden():
    z = np.load("tests/golden/scatter_adam.npz")
    grad = torch.zeros(53, 16, device=DEV)
    ops.scatter_add_sorted_(grad, g(torch.from_numpy(z["scatter.idx"])), g(torch.from_numpy(z["scatter.rows"])), None, 1.0, 0)
    got = grad.cpu().numpy()
    short = np.bincount(z["scatter.idx"], minlength=53) <= 64
    np.testing.assert_array_equal(got[short], z["scatter.grad"][short])  # torch's own embedding_dense_backward, bit for bit
    np.testing.assert_allclose(got[~short], z["scatter.grad"][~short], rtol=1e-5, atol=1e-5)  # >64 contributions: fixed piece tree
    np.testing.assert_array_equal(got, oc.embedding_grad_scatter_chunked(z["scatter.idx"], z["scatter.rows"], 53))


# -------------------------------------------------------------------------------------------- layernorm
@pytest.mark.parametrize("flavour", [L.LN_TORCH, L.LN_BERT])
@pytest.mark.parametrize("rows,d", [(7, 16), (33, 32), (1000, 64), (129, 128), (65, 256), (9, 512)])
def test_layernorm(flavour, rows, d):
    torch.manual_seed(rows + d)
    x = torch.randn(rows, d) * 2 + 0.5
    w, b = torch.randn(d), torch.randn(d)
    dy = torch.randn(rows, d)
    eps = 1e-8 if flavour == L.LN_TORCH else 1e-6
    xg, wg, bg = (g(t).requires_grad_(True) for t in (x, w, b))
    y = ops.layernorm(xg, wg, bg, eps, flavour)
    y.backward(g(dy))
    xr, wr, br = (t.clone().requires_grad_(True) for t in (x, w, b))
    ref = oc.torch_layernorm(xr, wr, br, eps) if flavour == L.LN_TORCH else oc.bert_layernorm(xr, wr, br, eps)
    ref.backward(dy)
    close(y, ref, 1e-5, 1e-5)
    close(xg.grad, xr.grad, 1e-4, 1e-5)
    close(wg.grad, wr.grad, 1e-4, 1e-4)
    close(bg.grad, br.grad, 1e-4, 1e-4)


# ----------------------------------------------------------------------------------------------- linear
def _ref_act(x, act):
    return {L.ACT_NONE: lambda t: t, L.ACT_RELU: torch.relu, L.ACT_GELU_TANH: oc.gelu_tanh}[act](x)


@pytest.mark.parametrize("M,N,K", [(10, 16, 16), (300, 192, 64), (257, 64, 256), (1000, 256, 64), (131, 48, 32),
                                   # weight block does not fit shared memory whole: column groups of the persistent kernel
                                   (1000, 128, 128), (700, 256, 128), (5000, 256, 128), (300, 1024, 256), (300, 256, 256),
                                   # K = 1024 / 768 at d = 256: split-K in 256-wide chunks (forward, and backward-data of the layers above)
                                   (300, 256, 1024), (260, 768, 256), (130, 512, 512)])
@pytest.mark.parametrize("act,res,rowtok,pA,pB", [(L.ACT_NONE, False, False, 0.0, 0.0), (L.ACT_GELU_TANH, False, False, 0.2, 0.0),
                                                  (L.ACT_NONE, True, False, 0.1, 0.3), (L.ACT_RELU, False, False, 0.2, 0.0),
                                                  (L.ACT_NONE, True, True, 0.2, 0.0)])
def test_linear(M, N, K, act, res, rowtok, pA, pB):
    torch.manual_seed(M + N)
    x, w, b = torch.randn(M, K), torch.randn(N, K) * 0.2, torch.randn(N)
    r = torch.randn(M, N) if res else None
    tok = (torch.rand(M) > 0.3).long() if rowtok else None
    dy = torch.randn(M, N)
    seed, sA, sB = 99, 3, 4
    xg, wg, bg = (g(t).requires_grad_(True) for t in (x, w, b))
    rg = g(r).requires_grad_(True) if res else None
    y = ops.linear(xg, wg, bg, residual=rg, row_tok=g(tok) if rowtok else None, act=act, pA=pA, siteA=sA, pB=pB, siteB=sB, seed=seed)
    y.backward(g(dy))
    xr, wr, br = (t.clone().requires_grad_(True) for t in (x, w, b))
    rr = r.clone().requires_grad_(True) if res else None
    ref = _ref_act(F.linear(xr, wr, br), act)
    if pA > 0:
        ref = ref * ops.dropout_mask(M * N, pA, seed, sA, DEV).cpu().view(M, N) / (1 - pA)
    if res:
        ref = ref + rr
    if pB > 0:
        ref = ref * ops.dropout_mask(M * N, pB, seed, sB, DEV).cpu().view(M, N) / (1 - pB)
    if rowtok:
        ref = ref * (tok != 0).unsqueeze(-1)
    ref.backward(dy)
    close(y, ref, 1e-4, 1e-4)
    close(xg.grad, xr.grad, 1e-4, 1e-4)
    acc = 1e-3 * max(1.0, math.sqrt(M / 1000.0))  # sums over M rows: the fp32 reference's own rounding grows with sqrt(M)
    close(wg.grad, wr.grad, 1e-4, acc)
    close(bg.grad, br.grad, 1e-4, acc)
    if res:
        close(rg.grad, rr.grad, 1e-5, 1e-5)


def test_linear_wide_many_tokens():
    """Wide layer over many tokens (several token slabs per dW tile in the split-fp16 weight-gradient kernel, several row tiles per
    CTA in the split-K forward / backward-data): plain Linear + bias (no ReLU: with 10^7 pre-activations a handful land within
    rounding of zero and flip their derivative in ANY implementation), against fp64."""
    torch.manual_seed(8)
    M, N, K = 20000, 512, 1024
    x, w, b = torch.randn(M, K, device=DEV), torch.randn(N, K, device=DEV) * 0.2, torch.randn(N, device=DEV)
    dy = torch.randn(M, N, device=DEV) * 1e-4  # gradient-sized values: the range scaling of the fp16 split must cope
    xg, wg, bg = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = ops.linear(xg, wg, bg)
    y.backward(dy)
    y64 = x.double() @ w.double().t() + b.double()
    dx64, dw64, db64 = dy.double() @ w.double(), dy.double().t() @ x.double(), dy.double().sum(0)
    rel = lambda a, r: float((a.detach().double() - r).abs().max() / r.abs().max())
    assert rel(y, y64) < 1e-5 and rel(xg.grad, dx64) < 1e-5, (rel(y, y64), rel(xg.grad, dx64))
    assert rel(wg.grad, dw64) < 1e-5 and rel(bg.grad, db64) < 1e-5, (rel(wg.grad, dw64), rel(bg.grad, db64))


def test_linear_strided_input():
    """q/k/v column blocks of a packed tensor are consumed through their row stride."""
    torch.manual_seed(1)
    big = torch.randn(50, 96)
    w = torch.randn(16, 32)
    y = ops.linear(g(big)[:, 32:64], g(w))
    close(y, F.linear(big[:, 32:64], w), 1e-4, 1e-4)


# -------------------------------------------------------------------------------------------- attention
def _ref_attention(q, k, v, tok, mode, scale, p, mask):
    s = torch.matmul(q, k.transpose(-2, -1)) * scale
    Ln = q.shape[-2]
    if mode == L.MASK_CAUSAL:
        s = s.masked_fill(~torch.tril(torch.ones(Ln, Ln, dtype=torch.bool)), float("-inf"))
    elif mode == L.MASK_KEYPAD:
        s = s.masked_fill((tok == 0)[:, None, None, :], -1e9)
    pr = F.softmax(s, dim=-1)
    if p > 0:
        pr = pr * mask / (1 - p)
    return torch.matmul(pr, v)


def _host_attn_mask(B, h, Ln, p, seed, site):
    """Keep mask [B, h, L, L] of an attention dropout site, computed on the host (oracle/common.py), not by the library."""
    return torch.from_numpy(oc.attn_keep_mask(B * h, Ln, p, seed, site)).view(B, h, Ln, Ln)


@pytest.mark.parametrize("B,Ln,h,dk", [(3, 8, 2, 8), (2, 13, 4, 8), (4, 50, 1, 64), (3, 50, 2, 64), (2, 200, 2, 32), (2, 200, 4, 64), (1, 256, 1, 16), (2, 100, 2, 128),
                                       (3, 37, 1, 64), (5, 64, 3, 64), (1, 1, 1, 64), (301, 50, 2, 64),
                                       (3, 129, 2, 64), (2, 256, 1, 64), (5, 65, 1, 64), (160, 200, 1, 64),
                                       # tcgen05 (d_k = 32): tile edges, one / two 128-query tiles, B*h*NT below and above 148 SMs
                                       (4, 1, 2, 32), (4, 15, 1, 32), (4, 16, 2, 32), (4, 17, 3, 32), (4, 100, 2, 32), (4, 127, 1, 32),
                                       (4, 128, 2, 32), (4, 129, 2, 32), (3, 255, 1, 32), (4, 256, 2, 32), (75, 128, 2, 32), (40, 256, 2, 32),
                                       # pair (d_k = 64, L <= 64): B*h odd and even (two items share one TMEM tile)
                                       (3, 1, 1, 64), (4, 2, 1, 64), (3, 33, 1, 64), (4, 63, 2, 64), (4, 64, 1, 64),
                                       # seq (d_k = 64, 64 < L <= 256)
                                       (4, 127, 2, 64), (4, 128, 1, 64), (3, 255, 1, 64),
                                       # SIMT head sizes
                                       (4, 30, 2, 24), (3, 45, 1, 40), (2, 129, 2, 40)])
@pytest.mark.parametrize("mode", [L.MASK_NONE, L.MASK_CAUSAL, L.MASK_KEYPAD])
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_attention_packed(B, Ln, h, dk, mode, p):
    """rbm_attn_fwd / rbm_attn_bwd on a packed q | k | v tensor against float64, dQ / dK / dV checked separately.  Sequence 0 is
    left-padded, 1 fully padded (softmax over -1e9 everywhere must stay finite / uniform), 2 has its last key as the only live
    key, the rest none."""
    torch.manual_seed(B * Ln + dk)
    d = h * dk
    qkv = torch.randn(B * Ln, 3 * d)
    tok = torch.randint(1, 50, (B, Ln))
    tok[0, : Ln // 3] = 0
    if B > 1:
        tok[1, :] = 0
    if B > 2:
        tok[2, :-1] = 0
    dout = torch.randn(B * Ln, d)
    scale = 1 / math.sqrt(dk)
    seed, site = 5, 11
    qg = g(qkv).requires_grad_(True)
    out = ops.attention(qg, None, g(tok), B, Ln, h, 0, d, 2 * d, mode, scale, p, seed, site)
    out.backward(g(dout))
    mask = _host_attn_mask(B, h, Ln, p, seed, site) if p > 0 else None
    if p > 0:
        assert abs(mask.float().mean().item() - (1 - p)) < 0.01 + 4 * math.sqrt(p * (1 - p) / mask.numel())
    qr = qkv.double().requires_grad_(True)
    q, k, v = (qr[:, i * d:(i + 1) * d].view(B, Ln, h, dk).transpose(1, 2) for i in range(3))
    ref = _ref_attention(q, k, v, tok, mode, scale, p, mask).transpose(1, 2).reshape(B * Ln, d)
    ref.backward(dout.double())
    close(out, ref, 1e-4, 1e-5)
    close(qg.grad[:, :d], qr.grad[:, :d], 1e-3, 2e-5, "dq")
    close(qg.grad[:, 2 * d:], qr.grad[:, 2 * d:], 1e-3, 2e-5, "dv")
    # dK_j = scale * sum_i P_ij (dP_ij - delta_i) q_i cancels: for the only live key of a sequence (P = 1 from every query) it is
    # exactly 0 while each of its L terms carries fp32 rounding of dP and delta.  The bar is 2e-5 plus 4 ulp of the sum of the
    # terms' magnitudes (below 1e-6 for a key that shares the softmax with others).
    with torch.no_grad():
        s = (q @ k.transpose(-1, -2)) * scale
        if mode == L.MASK_CAUSAL:
            s = s.masked_fill(~torch.tril(torch.ones(Ln, Ln, dtype=torch.bool)), float("-inf"))
        elif mode == L.MASK_KEYPAD:
            s = s.masked_fill((tok == 0)[:, None, None, :], -1e9)
        pr = torch.softmax(s, -1) * (mask / (1 - p) if p > 0 else 1.0)
        dp = dout.double().view(B, Ln, h, dk).transpose(1, 2) @ v.transpose(-1, -2)
        mag = scale * ((pr * dp).abs().transpose(-1, -2) @ q.abs()).transpose(1, 2).reshape(B * Ln, d)
    err = (qg.grad[:, d:2 * d].cpu().double() - qr.grad[:, d:2 * d]).abs()
    bound = 1e-3 * qr.grad[:, d:2 * d].abs() + 2e-5 + 2.4e-7 * mag
    assert bool((err <= bound).all()), ("dk", float((err - bound).max()), float(err.max()))


@pytest.mark.skipif(os.environ.get("RBM_ATTN_IMPL") == "mma", reason="rbm_attn_fwd_lq / _bwd_lq exist on the tensor path only")
@pytest.mark.parametrize("B,Ln,Lq,h", [(5, 200, 48, 2), (90, 200, 32, 2), (3, 200, 128, 1), (7, 130, 16, 2), (2, 256, 144, 2), (4, 40, 16, 2)])
@pytest.mark.parametrize("mode", [L.MASK_NONE, L.MASK_KEYPAD])
@pytest.mark.parametrize("p", [0.0, 0.15])
def test_attention_compacted_queries(B, Ln, Lq, h, mode, p):
    """rbm_attn_fwd_lq / rbm_attn_bwd_lq (Lq query rows per sequence against all L keys; the final block of BERT4Rec training needs
    the labelled positions' queries only) against the same reference with the host-side Philox mask: the dropout stream is
    indexed by (sequence-head, query ordinal, key), i.e. the first Lq rows of the [L x L] mask."""
    torch.manual_seed(B * Ln + Lq)
    dk = 32
    d = h * dk
    q = torch.randn(B * Lq, d)
    nreal = torch.randint(0, Lq + 1, (B,))
    nreal[0] = Lq
    for b in range(B):
        q[b * Lq + int(nreal[b]): (b + 1) * Lq] = 0  # the zero rows that pad a sequence's queries
    kv = torch.randn(B * Ln, 2 * d)
    tok = torch.randint(1, 50, (B, Ln))
    tok[0, : Ln // 3] = 0
    if B > 1:
        tok[1, :] = 0
    dout = torch.randn(B * Lq, d)
    for b in range(B):
        dout[b * Lq + int(nreal[b]): (b + 1) * Lq] = 0
    scale = 1 / math.sqrt(dk)
    seed, site = 7, 13
    qg, kvg = g(q).requires_grad_(True), g(kv).requires_grad_(True)
    out = ops.attention_lq(qg, kvg, g(tok), B, Ln, Lq, h, mode, scale, p, seed, site)
    out.backward(g(dout))
    mask = _host_attn_mask(B, h, Ln, p, seed, site)[:, :, :Lq, :] if p > 0 else None
    qr, kvr = q.clone().requires_grad_(True), kv.clone().requires_grad_(True)
    qq = qr.view(B, Lq, h, dk).transpose(1, 2).double()
    kk, vv = (kvr[:, i * d:(i + 1) * d].view(B, Ln, h, dk).transpose(1, 2).double() for i in range(2))
    sc = qq @ kk.transpose(-1, -2) * scale
    if mode == L.MASK_KEYPAD:
        sc = sc.masked_fill((tok == 0)[:, None, None, :], -1e9)
    pr = torch.softmax(sc, -1)
    if p > 0:
        pr = pr * mask.double() / (1 - p)
    ref = (pr @ vv).transpose(1, 2).reshape(B * Lq, d)
    ref.backward(dout.double())
    close(out, ref.float(), 1e-4, 1e-5)
    close(qg.grad, qr.grad, 1e-3, 2e-5)
    close(kvg.grad, kvr.grad, 1e-3, 2e-5)


@pytest.mark.parametrize("mode", [L.MASK_CAUSAL, L.MASK_KEYPAD])
def test_attention_persistent_many_items(mode):
    """More (sequence, head, tile) work items than SMs: every persistent tcgen05 CTA walks several items, so the
    cross-item hand-shakes (operand staging, accumulator hand-back, ring phases) are on the tested path."""
    torch.manual_seed(7)
    B, Ln, h, dk, p = 90, 200, 2, 32, 0.1
    d = h * dk
    qkv = torch.randn(B * Ln, 3 * d)
    tok = torch.randint(1, 50, (B, Ln))
    tok[::3, : Ln // 4] = 0
    tok[5, :] = 0
    tok[5, -1] = 5 if mode == L.MASK_CAUSAL else 0
    dout = torch.randn(B * Ln, d)
    scale = 1 / math.sqrt(dk)
    seed, site = 9, 3
    qg = g(qkv).requires_grad_(True)
    out = ops.attention(qg, None, g(tok), B, Ln, h, 0, d, 2 * d, mode, scale, p, seed, site)
    out.backward(g(dout))
    mask = _host_attn_mask(B, h, Ln, p, seed, site)
    qr = qkv.clone().requires_grad_(True)
    q, k, v = (qr[:, i * d:(i + 1) * d].view(B, Ln, h, dk).transpose(1, 2) for i in range(3))
    ref = _ref_attention(q, k, v, tok, mode, scale, p, mask).transpose(1, 2).reshape(B * Ln, d)
    ref.backward(dout)
    close(out, ref, 1e-4, 1e-5)
    close(qg.grad, qr.grad, 1e-3, 2e-5)


def test_attention_split_sources_and_bad_shapes():
    torch.manual_seed(0)
    B, Ln, h, dk = 2, 20, 2, 16
    d = h * dk
    q, kv = torch.randn(B * Ln, d), torch.randn(B * Ln, 2 * d)
    dout = torch.randn(B * Ln, d)
    qg, kvg = g(q).requires_grad_(True), g(kv).requires_grad_(True)
    out = ops.attention(qg, kvg, None, B, Ln, h, 0, 0, d, L.MASK_CAUSAL, 0.25)
    out.backward(g(dout))
    qr, kvr = q.clone().requires_grad_(True), kv.clone().requires_grad_(True)
    sp = lambda t: t.view(B, Ln, h, dk).transpose(1, 2)
    ref = _ref_attention(sp(qr), sp(kvr[:, :d]), sp(kvr[:, d:]), None, L.MASK_CAUSAL, 0.25, 0.0, None).transpose(1, 2).reshape(B * Ln, d)
    ref.backward(dout)
    close(out, ref, 1e-4, 1e-5)
    close(qg.grad, qr.grad, 1e-3, 2e-5)
    close(kvg.grad, kvr.grad, 1e-3, 2e-5)
    with pytest.raises(RuntimeError):  # L > 256 is unsupported and must say so
        ops.attention(g(torch.randn(300, 48)), None, None, 1, 300, 1, 0, 16, 32, L.MASK_CAUSAL, 1.0)


# ----------------------------------------------------------------------------------- scoring + cross-entropy
@pytest.mark.parametrize("n,V1,d,frac", [(40, 38, 16, 0.5), (500, 3417, 64, 0.15), (300, 1001, 128, 0.3), (130, 777, 256, 0.9), (64, 65, 32, 0.0),
                                          (700, 64, 128, 0.4), (3000, 5003, 256, 0.2), (520, 20011, 256, 0.3), (64, 300, 256, 0.0),
                                          (900, 12101, 128, 0.15)])
def test_score_ce(n, V1, d, frac):
    torch.manual_seed(n)
    h = torch.randn(n, d)
    w, b = torch.randn(V1, d) * 0.3, torch.randn(V1)
    labels = torch.where(torch.rand(n) < frac, torch.randint(1, V1, (n,)), torch.zeros(n, dtype=torch.long))
    if frac == 0.0:
        labels[5] = V1 - 1  # exactly one scored row, last vocabulary id
    hg, wg, bg = (g(t).requires_grad_(True) for t in (h, w, b))
    loss = ops.score_cross_entropy(hg, g(labels), wg, bg)
    (loss * 1.7).backward()
    hr, wr, br = (t.clone().requires_grad_(True) for t in (h, w, b))
    ref = F.cross_entropy(F.linear(hr, wr, br), labels, ignore_index=0)
    (ref * 1.7).backward()
    assert abs(loss.item() - ref.item()) < 1e-5 * max(1.0, abs(ref.item()))
    close(hg.grad, hr.grad, 1e-3, 1e-6)
    close(wg.grad, wr.grad, 1e-3, 1e-6)
    close(bg.grad, br.grad, 1e-3, 1e-6)


# -------------------------------------------------------------------------------------- SAS scoring + BCE
@pytest.mark.parametrize("rows,d,V", [(30, 16, 20), (1000, 64, 3417), (640, 128, 12102)])
def test_sas_score_bce(rows, d, V):
    torch.manual_seed(rows)
    f, table = torch.randn(rows, d), torch.randn(V, d) * 0.3
    table[0] = 0
    pos = torch.randint(0, V, (rows,))
    pos[::3] = 0
    neg = torch.randint(0, V, (rows,))
    fg, tg = g(f).requires_grad_(True), g(table).requires_grad_(True)
    pl, nl = ops.sas_scores(fg, tg, g(pos), g(neg))
    loss = ops.bce_pair_loss(pl, nl, g(pos))
    loss.backward()
    fr, tr = f.clone().requires_grad_(True), table.clone().requires_grad_(True)
    plr = (fr * F.embedding(pos, tr, padding_idx=0)).sum(-1)
    nlr = (fr * F.embedding(neg, tr, padding_idx=0)).sum(-1)
    idx = pos != 0
    ref = F.binary_cross_entropy_with_logits(plr[idx], torch.ones(int(idx.sum()))) + \
        F.binary_cross_entropy_with_logits(nlr[idx], torch.zeros(int(idx.sum())))
    ref.backward()
    close(pl, plr, 1e-4, 1e-5)
    close(nl, nlr, 1e-4, 1e-5)
    assert abs(loss.item() - ref.item()) < 1e-5 * max(1.0, abs(ref.item()))
    close(fg.grad, fr.grad, 1e-4, 1e-7)
    close(tg.grad, tr.grad, 1e-4, 1e-7)


def test_candidate_scores():
    torch.manual_seed(0)
    U, Cn, d, V = 9, 101, 64, 500
    f3 = torch.randn(U, 7, d)
    table, bias = torch.randn(V, d), torch.randn(V)
    cand = torch.randint(0, V, (U, Cn))
    out = ops.candidate_scores(g(f3)[:, -1, :], g(table), g(bias), g(cand))
    ref = torch.einsum("ucd,ud->uc", table[cand], f3[:, -1, :]) + bias[cand]
    close(out, ref, 1e-4, 1e-5)


# ------------------------------------------------------------------------------------------------ top-k
@pytest.mark.parametrize("U,Cn,k", [(5, 101, 10), (17, 3416, 10), (3, 40, 20), (4, 7, 10), (2, 100000, 32)])
def test_topk_rows_bit_exact_with_ties(U, Cn, k):
    rng = np.random.RandomState(U * Cn)
    scores = rng.randn(U, Cn).astype(np.float32)
    scores[:, Cn // 2:] = np.round(scores[:, Cn // 2:], 1)  # plenty of exact ties
    scores[0, :] = 1.0  # all tied: ids must come out ascending
    ref_v, ref_i = om.topk_canonical(scores, k, id_offset=3)
    v, i = ops.topk_rows(g(torch.from_numpy(scores)), k, id_offset=3)
    np.testing.assert_array_equal(i.cpu().numpy(), ref_i)
    np.testing.assert_array_equal(v.cpu().numpy(), ref_v)


@pytest.mark.parametrize("U,V,d,k,bias", [(10, 300, 16, 10, False), (70, 3416, 64, 10, True), (130, 12101, 128, 10, False), (64, 5000, 256, 20, True),
                                          (200, 40000, 64, 10, True), (33, 9000, 32, 16, False)])
def test_score_topk_fused(U, V, d, k, bias):
    """ids AND scores equal to the canonical top-k of the fp32 scores (sequential-FMA contract, oracle/metrics.py) on every row:
    the fp32 scan kernel, the tcgen05 selection + exact re-score (catalogues >= 8192 items, k <= 10), and the same with every
    user forced through the exact re-scan (stage 3)."""
    import os
    torch.manual_seed(U + V)
    f, table = torch.randn(U, d), torch.randn(V + 1, d)
    b = torch.randn(V + 1) if bias else None
    sc = om.scores_fp32_sequential(g(f), g(table[1:]), g(b[1:]) if bias else None).cpu().numpy()
    ref_v, ref_i = om.topk_canonical(sc, k, id_offset=1)
    for eps in (None, "1e9"):
        if eps:
            os.environ["RBM_TOPK_EPS"] = eps
        try:
            vals, ids = ops.score_topk(g(f), g(table), g(b) if bias else None, 1, V + 1, k)
        finally:
            os.environ.pop("RBM_TOPK_EPS", None)
        np.testing.assert_array_equal(ids.cpu().numpy(), ref_i)
        np.testing.assert_array_equal(vals.cpu().numpy(), ref_v)


def test_score_topk_adversarial_near_ties():
    """Catalogue built so that thousands of items sit within the TF32 error of each user's k-th best score: the approximate
    candidate lists cannot contain the right answer, the certificate must notice and the exact re-scan must deliver it."""
    torch.manual_seed(5)
    U, V, d, k = 96, 20000, 64, 10
    f = torch.randn(U, d)
    base = torch.randn(d)
    table = base.unsqueeze(0) * (1.0 + 1e-5 * torch.randn(V + 1, 1)) + 1e-5 * torch.randn(V + 1, d)  # all items nearly collinear
    sc = om.scores_fp32_sequential(g(f), g(table[1:])).cpu().numpy()
    ref_v, ref_i = om.topk_canonical(sc, k, id_offset=1)
    vals, ids = ops.score_topk(g(f), g(table), None, 1, V + 1, k)
    np.testing.assert_array_equal(ids.cpu().numpy(), ref_i)
    np.testing.assert_array_equal(vals.cpu().numpy(), ref_v)


def test_topk_merge_shard_invariance():
    rng = np.random.RandomState(3)
    U, V, k = 33, 4000, 10
    scores = np.round(rng.randn(U, V).astype(np.float32), 2)  # ties across shards
    ref_v, ref_i = om.topk_canonical(scores, k, id_offset=1)
    sg = g(torch.from_numpy(scores))
    for S in (1, 2, 3, 8):
        bounds = np.linspace(0, V, S + 1).astype(int)
        parts = [ops.topk_rows(sg[:, a:b2], k, id_offset=1 + int(a)) for a, b2 in zip(bounds[:-1], bounds[1:])]
        v, i = ops.topk_merge(torch.stack([p[0] for p in parts]), torch.stack([p[1] for p in parts]))
        np.testing.assert_array_equal(i.cpu().numpy(), ref_i)
        np.testing.assert_array_equal(v.cpu().numpy(), ref_v)


def test_metrics_match_reference_golden():
    z = np.load("tests/golden/metrics.npz")
    for tag, ks in (("c101", [1, 5, 10, 20]), ("c3416", [1, 5, 10, 20]), ("multi", [1, 5, 10])):
        scores, labels = torch.from_numpy(z[tag + ".scores"]), torch.from_numpy(z[tag + ".labels"])
        m = rbm_b200.recalls_ndcgs_and_mrr_for_ks(g(scores), g(labels), ks)
        keys = [str(k) for k in z[tag + ".keys"]]
        assert sorted(m.keys()) == keys
        got = np.array([m[k] for k in keys])
        np.testing.assert_allclose(got, z[tag + ".vals"], rtol=2e-6, atol=1e-7)
        if tag != "multi":  # per-user values and HR are bit-exact
            _, ids = ops.topk_rows(g(scores), 20)
            np.testing.assert_array_equal(ids.cpu().numpy(), z[tag + ".rank20"])
            pu = ops.rank_metrics(ids, [20, 10, 5, 1], labels=g(labels)).cpu().numpy()
            ref = om.recalls_ndcgs_and_mrr_for_ks(scores, labels, ks, per_user=True)
            for j, k in enumerate([20, 10, 5, 1]):
                np.testing.assert_array_equal(pu[:, j, 0], ref["Recall@%d" % k].numpy())
                np.testing.assert_array_equal(pu[:, j, 1], ref["NDCG@%d" % k].numpy())
                np.testing.assert_array_equal(pu[:, j, 2], ref["MRR@%d" % k].numpy())
            pu2 = ops.rank_metrics(ids, [10], positives=g(torch.zeros(scores.shape[0], dtype=torch.long))).cpu().numpy()
            np.testing.assert_array_equal(pu2[:, 0, 1], ref["NDCG@10"].numpy())


# ------------------------------------------------------------------------------------------------- Adam
def test_fused_adam_matches_torch_golden():
    z = np.load("tests/golden/scatter_adam.npz")
    p = torch.nn.Parameter(g(torch.from_numpy(z["adam.p0"])))
    odd = torch.nn.Parameter(g(torch.randn(4097 * 3 + 1)))  # multi-chunk, ragged tail
    odd_ref = odd.detach().cpu().numpy().copy()
    m_ref, v_ref = np.zeros_like(odd_ref), np.zeros_like(odd_ref)
    opt = rbm_b200.FusedAdam([p, odd], lr=1e-3)
    rng = np.random.RandomState(0)
    for s in range(4):
        p.grad = g(torch.from_numpy(z["adam.grads"][s].copy()))
        go = rng.randn(odd_ref.size).astype(np.float32)
        odd.grad = g(torch.from_numpy(go))
        opt.step()
        np.testing.assert_allclose(p.detach().cpu().numpy(), z["adam.ps"][s], rtol=1e-6, atol=1e-7)
        oo.adam_step(odd_ref, go, m_ref, v_ref, s + 1, 1e-3)
        np.testing.assert_allclose(odd.detach().cpu().numpy(), odd_ref, rtol=1e-5, atol=1e-7)
    st = opt.state[p]
    np.testing.assert_allclose(st["exp_avg"].cpu().numpy(), z["adam.m"], rtol=1e-5, atol=1e-8)
    np.testing.assert_allclose(st["exp_avg_sq"].cpu().numpy(), z["adam.v"], rtol=1e-5, atol=1e-12)
    assert set(opt.state_dict()["state"][0].keys()) == {"step", "exp_avg", "exp_avg_sq"}


# ------------------------------------------------------------------------- device-side batch construction
def _csr(hist):
    ptr = np.cumsum([0] + [len(h) for h in hist]).astype(np.int64)
    items = np.array([i for h in hist for i in h], np.int64)
    return g(torch.from_numpy(ptr)), g(torch.from_numpy(items))


def test_batch_construction_golden():
    """The kernels reproduce what the REFERENCE dataloaders produce when fed the contract's random numbers
    (tests/golden/batches.npz, minted by driving BertTrainDataset / sample_function with injected Philox words)."""
    import os
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "batches.npz"))
    ptr, items = g(torch.from_numpy(z["hist_ptr"])), g(torch.from_numpy(z["hist_items"]))
    V, seed = int(z["num_items"]), int(z["seed"])
    step = int(z["site"]) - ops.BATCH_SITE_BASE
    for tag, Ln in [("bert_L8", 8), ("bert_L16_all", 16), ("bert_L8_none", 8)]:
        t, l = ops.bert_cloze_batch(ptr, items, g(torch.from_numpy(z[tag + ".users"])), Ln, float(z[tag + ".mask_prob"]), V + 1, V, seed, step)
        np.testing.assert_array_equal(t.cpu().numpy(), z[tag + ".tokens"])
        np.testing.assert_array_equal(l.cpu().numpy(), z[tag + ".labels"])
    for tag, Ln in [("sas_L8", 8), ("sas_L50", 50)]:
        s, p, n = ops.sas_train_batch(ptr, items, g(torch.from_numpy(z[tag + ".users"])), Ln, V, seed, step)
        np.testing.assert_array_equal(s.cpu().numpy(), z[tag + ".seq"])
        np.testing.assert_array_equal(p.cpu().numpy(), z[tag + ".pos"])
        np.testing.assert_array_equal(n.cpu().numpy(), z[tag + ".neg"])


@pytest.mark.parametrize("Ln,V", [(50, 60), (200, 3416), (256, 300)])
def test_batch_construction_ragged_vs_oracle(Ln, V):
    """Empty, one-item, short, exactly-L and longer-than-L histories, repeated items, a user who owns (almost) every item."""
    from oracle import batches as obt
    rs = np.random.RandomState(Ln + V)
    lens = [0, 1, 2, 3, Ln - 1, Ln, Ln + 1, 2 * Ln + 7] + list(rs.randint(2, 3 * Ln, size=40))
    hist = [list(rs.randint(1, V + 1, size=n)) for n in lens]
    hist.append(list(range(1, V + 1))[-Ln:])          # a window that covers a contiguous block of ids
    hist.append([7] * (Ln + 3))                        # one item repeated
    users = list(rs.randint(0, len(hist), size=64)) + list(range(len(hist)))
    ptr, items = _csr(hist)
    ug = g(torch.tensor(users, dtype=torch.int64))
    seed, step = 99, 12
    t, l = ops.bert_cloze_batch(ptr, items, ug, Ln, 0.15, V + 1, V, seed, step)
    to, lo = obt.bert_cloze_batch(hist, users, Ln, 0.15, V + 1, V, seed, ops.BATCH_SITE_BASE + step)
    np.testing.assert_array_equal(t.cpu().numpy(), to)
    np.testing.assert_array_equal(l.cpu().numpy(), lo)
    s, p, n = ops.sas_train_batch(ptr, items, ug, Ln, V, seed, step)
    so, po, no = obt.sas_train_batch(hist, users, Ln, V, seed, ops.BATCH_SITE_BASE + step)
    np.testing.assert_array_equal(s.cpu().numpy(), so)
    np.testing.assert_array_equal(p.cpu().numpy(), po)
    np.testing.assert_array_equal(n.cpu().numpy(), no)


def test_batch_construction_properties_at_bench_size():
    """cfg2-sized batch (B=1024, L=200): rates of the 15 % / 80-10-10 rule, structural invariants, determinism."""
    rs = np.random.RandomState(5)
    V, U, Ln, Bsz = 3416, 2000, 200, 1024
    hist = [list(rs.randint(1, V + 1, size=n)) for n in rs.randint(20, 400, size=U)]
    ptr, items = _csr(hist)
    users = g(torch.from_numpy(rs.randint(0, U, size=Bsz).astype(np.int64)))
    t, l = ops.bert_cloze_batch(ptr, items, users, Ln, 0.15, V + 1, V, 3, 0)
    t2, l2 = ops.bert_cloze_batch(ptr, items, users, Ln, 0.15, V + 1, V, 3, 0)
    assert torch.equal(t, t2) and torch.equal(l, l2)
    t3, _ = ops.bert_cloze_batch(ptr, items, users, Ln, 0.15, V + 1, V, 3, 1)
    assert not torch.equal(t, t3)  # another step, another mask
    t, l = t.cpu(), l.cpu()
    real = torch.zeros_like(t, dtype=torch.bool)
    for b, u in enumerate(users.cpu().tolist()):
        n = min(len(hist[u]), Ln)
        real[b, Ln - n:] = True
        assert torch.equal(torch.where(l[b] != 0, l[b], t[b])[Ln - n:], torch.tensor(hist[u][-n:]))  # unmasked view = history
    assert (t[~real] == 0).all() and (l[~real] == 0).all()
    scored = (l != 0) & real
    rate = scored.float().sum() / real.float().sum()
    assert abs(rate - 0.15) < 0.005
    masked = (t == V + 1) & scored
    assert abs(masked.float().sum() / scored.float().sum() - 0.8) < 0.02
    kept = (t == l) & scored
    assert abs(kept.float().sum() / scored.float().sum() - 0.1) < 0.02  # + 1/V of the random replacements
    s, p, n = (x.cpu() for x in ops.sas_train_batch(ptr, items, users, 50, V, 3, 0))
    assert torch.equal(s[:, 1:][p[:, :-1] != 0], p[:, :-1][p[:, :-1] != 0])  # pos is seq shifted by one
    for b, u in enumerate(users.cpu().tolist()[:64]):
        w = set(hist[u][-50:])
        assert all(int(x) not in w for x in n[b][p[b] != 0].tolist())
    assert (n[p == 0] == 0).all() and (n <= V).all() and (n >= 0).all()


# ------------------------------------------------------------------------------------ evaluation negatives / batches
def _gold_split(z, name):
    ptr, items = z[name + "_ptr"], z[name + "_items"]
    return [items[ptr[u]:ptr[u + 1]].tolist() for u in range(len(ptr) - 1)]


def test_negative_samples_and_eval_batch_golden():
    """rbm_negative_samples / rbm_eval_batch reproduce what the REFERENCE samplers and eval datasets produce when fed the
    contract's random numbers (tests/golden/eval_batches.npz); also through the loader classes."""
    import os
    from rbm_b200.dataloaders import DeviceNegativeSampler, DeviceEvalLoader
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "eval_batches.npz"))
    tr, va, te = _gold_split(z, "train"), _gold_split(z, "val"), _gold_split(z, "test")
    V, S, seed = int(z["num_items"]), int(z["sample_size"]), int(z["seed"])
    assert int(z["site"]) == ops.NEG_SITE
    negs = {}
    for code in ("random", "popular"):
        smp = DeviceNegativeSampler(tr, va, te, len(tr), V, S, seed, DEV, code=code)
        negs[code] = smp.get_negative_samples()
        np.testing.assert_array_equal(negs[code].cpu().numpy(), z["neg_" + code])
        part = ops.negative_samples(smp.seen_ptr, smp.seen_items, V, S, seed, smp.cdf, user_begin=3, num_users=4)
        np.testing.assert_array_equal(part.cpu().numpy(), z["neg_" + code][3:7])
    for model, mask in (("bert", V + 1), ("sas", -1)):
        for Ln in (8, 16):
            ld = DeviceEvalLoader(tr, va, negs["random"], Ln, 4, DEV, mask_token=mask)
            parts = list(ld)
            assert len(parts) == len(ld) == 3
            for j, nm in enumerate(("seq", "cand", "labels")):
                got = torch.cat([p[j] for p in parts]).cpu().numpy()
                np.testing.assert_array_equal(got, z["%s_L%d.%s" % (model, Ln, nm)])


@pytest.mark.parametrize("V,U,S", [(300, 500, 100), (3416, 2000, 100), (40, 64, 8)])
def test_negative_samples_ragged_vs_oracle(V, U, S):
    """Empty seen sets, users who have seen most of the catalogue, heavy-tailed popularity; bit-exact vs the oracle."""
    from oracle import batches as obt
    rs = np.random.RandomState(V + U)
    lens = np.minimum(rs.randint(0, max(2, V // 2), size=U), V - S - 1)
    lens[0], lens[1] = 0, V - S  # nothing seen / exactly S unseen items left
    seen = [sorted(rs.choice(V, size=n, replace=False) + 1) for n in lens]
    counts = np.maximum(1, (1000.0 / np.arange(1, V + 1)).astype(np.int64))
    counts[rs.permutation(V)[: V // 10]] = 0  # items nobody interacted with are never drawn by popularity
    ptr, items = _csr(seen)
    cdf = g(torch.from_numpy(np.cumsum(counts)))
    nu = 48 if V > 1000 else U  # the pure-python oracle is slow: a user sub-range at the larger sizes
    for code, c, pc in (("random", None, None), ("popular", cdf, counts.tolist())):
        out = ops.negative_samples(ptr, items, V, S, 77, c, user_begin=0, num_users=nu).cpu().numpy()
        ref = obt.negative_samples(seen, V, S, 77, ops.NEG_SITE, pop_counts=pc, user_begin=0, num_users=nu)
        np.testing.assert_array_equal(out, ref)
        full = ops.negative_samples(ptr, items, V, S, 77, c).cpu().numpy()
        np.testing.assert_array_equal(full[:nu], out)
        for u in range(U):
            row = full[u][full[u] >= 0].tolist()
            assert len(set(row)) == len(row) and not (set(row) & set(int(i) for i in seen[u]))
            if code == "random":
                assert len(row) == S


def test_eval_batch_ragged_vs_oracle():
    from oracle import batches as obt
    rs = np.random.RandomState(3)
    V, Ln, N = 500, 50, 100
    lens = [0, 1, Ln - 1, Ln, Ln + 1, 3 * Ln] + list(rs.randint(0, 120, size=60))
    hist = [list(rs.randint(1, V + 1, size=n)) for n in lens]
    U = len(hist)
    answers = rs.randint(1, V + 1, size=U).astype(np.int64)
    negatives = rs.randint(1, V + 1, size=(U, N)).astype(np.int64)
    users = list(rs.permutation(U)) + [0, 0, 5]
    ptr, items = _csr(hist)
    for mask in (V + 1, -1):
        s, c, l = ops.eval_batch(ptr, items, g(torch.from_numpy(answers)), g(torch.from_numpy(negatives)),
                                 g(torch.tensor(users, dtype=torch.int64)), Ln, mask)
        so, co, lo = obt.eval_batch(hist, answers, negatives, users, Ln, mask)
        np.testing.assert_array_equal(s.cpu().numpy(), so)
        np.testing.assert_array_equal(c.cpu().numpy(), co)
        np.testing.assert_array_equal(l.cpu().numpy(), lo)


def test_score_topk_full_size_properties():
    """Full-catalogue scoring + top-10 at a BASELINE-sized catalogue (10^6 items, ragged end, bias): sorted scores, distinct
    in-range ids, ids and scores IDENTICAL to the canonical top-k of the fp32 scores (oracle/metrics.scores_fp32_sequential) on
    a sample of users, the set equal to an fp64 ranking wherever the k-th gap is clear, and exact shard-count invariance (two
    half-catalogue calls merged == one call, every row); k = 16 (exact fp32 scan path) against the same oracle."""
    torch.manual_seed(7)
    U, V, d, k = 1024, 1_000_003, 64, 10
    f = torch.randn(U, d, device=DEV)
    table = torch.randn(V + 1, d, device=DEV)
    b = torch.randn(V + 1, device=DEV)
    vals, ids = ops.score_topk(f, table, b, 1, V + 1, k)
    assert bool((vals[:, :-1] >= vals[:, 1:]).all())
    assert int(ids.min()) >= 1 and int(ids.max()) <= V
    assert all(len(set(r)) == k for r in ids[:64].tolist()) and int((ids.sort(1).values.diff(dim=1) == 0).sum()) == 0
    n = 128
    sc32 = om.scores_fp32_sequential(f[:n], table[1:], b[1:])
    rv32, ri32 = torch.topk(sc32, 16, dim=1)  # no exact ties among the top scores of random data: topk == canonical order
    assert bool((rv32[:, :-1] > rv32[:, 1:]).all())
    assert torch.equal(ids[:n], ri32[:, :k] + 1)
    assert torch.equal(vals[:n], rv32[:, :k])
    sc = f[:n].double() @ table[1:].double().t() + b[1:].double()
    rv, ri = torch.topk(sc, k + 1, dim=1)
    clear = (rv[:, k - 1] - rv[:, k]) > 1e-3  # k-th and (k+1)-th score apart by more than fp32 noise: the SET is determined
    got, ref = ids[:n].sort(1).values, (ri[:, :k] + 1).sort(1).values
    assert bool((got[clear] == ref[clear]).all()) and float(clear.float().mean()) > 0.9
    half = 1 + V // 2
    v1, i1 = ops.score_topk(f, table, b, 1, half, k)
    v2, i2 = ops.score_topk(f, table, b, half, V + 1, k)
    mv, mi = ops.topk_merge(torch.stack([v1, v2]), torch.stack([i1, i2]))
    assert torch.equal(mi, ids) and torch.equal(mv, vals)
    v16, i16 = ops.score_topk(f[:64], table, b, 1, V + 1, 16)
    assert torch.equal(i16, ri32[:64] + 1) and torch.equal(v16, rv32[:64])


def _ce_ref64(h, labels, w, b, chunk=65536):
    """fp64 torch evaluation of the masked cross-entropy and its gradients, chunked over the vocabulary (on the device the
    tensors live on): loss, dH [n, d] (zeros at ignored rows), dW, db."""
    sel = labels != 0
    hc, tg = h[sel].double(), labels[sel]
    V1 = w.shape[0]
    lse = torch.full((hc.shape[0],), -float("inf"), dtype=torch.float64, device=h.device)
    for v0 in range(0, V1, chunk):
        lg = hc @ w[v0:v0 + chunk].double().t() + b[v0:v0 + chunk].double()
        lse = torch.logaddexp(lse, torch.logsumexp(lg, 1))
    tl = (hc * w[tg].double()).sum(1) + b[tg].double()
    P = hc.shape[0]
    dh_c = torch.zeros_like(hc)
    dw = torch.zeros(V1, w.shape[1], dtype=torch.float64, device=h.device)
    db = torch.zeros(V1, dtype=torch.float64, device=h.device)
    for v0 in range(0, V1, chunk):
        wc = w[v0:v0 + chunk].double()
        G = torch.exp(hc @ wc.t() + b[v0:v0 + chunk].double() - lse[:, None])
        inb = (tg >= v0) & (tg < v0 + chunk)
        G[inb.nonzero(as_tuple=True)[0], tg[inb] - v0] -= 1.0
        G /= P
        dh_c += G @ wc
        dw[v0:v0 + chunk] = G.t() @ hc
        db[v0:v0 + chunk] = G.sum(0)
    dh = torch.zeros(h.shape, dtype=torch.float64, device=h.device)
    dh[sel] = dh_c
    return float((lse - tl).mean()), dh, dw, db


@pytest.mark.parametrize("passes", [3, 1])
def test_score_ce_wide_million_items(passes):
    """BASELINE configs[3] scoring shape: d = 256 over 10^6 + 1 output rows (split-fp16 tcgen05 kernels, csrc/ce_wide.cu) against
    an fp64 evaluation: loss 1e-6 relative, dH / dW / db 1e-4 of their scale in the default three-pass (fp32-parity) mode; the
    single-pass fp16 mode (RBM_CE_WIDE_PASSES=1, the optional reduced-precision line) stays within the north star's 1e-3."""
    import os
    torch.manual_seed(3)
    n, V1, d = 6000, 1_000_001, 256
    h = (torch.randn(n, d, device=DEV) * 0.5).requires_grad_(True)
    w = (torch.randn(V1, d, device=DEV) * 0.05).requires_grad_(True)
    b = (torch.randn(V1, device=DEV) * 0.1).requires_grad_(True)
    labels = torch.where(torch.rand(n, device=DEV) < 0.15, torch.randint(1, V1, (n,), device=DEV), torch.zeros(n, dtype=torch.long, device=DEV))
    labels[7], labels[8] = V1 - 1, 1
    os.environ["RBM_CE_WIDE_PASSES"] = str(passes)
    try:
        loss = ops.score_cross_entropy(h, labels, w, b)
        loss.backward()
        torch.cuda.synchronize()
    finally:
        os.environ.pop("RBM_CE_WIDE_PASSES", None)
    rl, rdh, rdw, rdb = _ce_ref64(h.detach(), labels, w.detach(), b.detach())
    tol_l, tol_g = (1e-6, 1e-4) if passes == 3 else (1e-4, 1e-3)
    assert abs(loss.item() - rl) < tol_l * abs(rl), (loss.item(), rl)
    for got, ref, name in ((h.grad, rdh, "dH"), (w.grad, rdw, "dW"), (b.grad, rdb, "db")):
        err = float((got.double() - ref).abs().max() / ref.abs().max())
        assert err < tol_g, (name, err)
    assert float(b.grad.sum().abs()) < 1e-5 and float(w.grad.sum(0).abs().max()) < 1e-5  # rows of softmax - onehot sum to zero


def test_score_ce_wide_range_scaling():
    """The split-fp16 path range-scales both operands by per-tensor powers of two: hidden states of magnitude 1e3 against weights
    of magnitude 1e-4 (and the reverse) keep fp32-level accuracy; nothing overflows fp16."""
    for hs, ws in ((1e3, 1e-4), (1e-3, 50.0)):
        torch.manual_seed(5)
        n, V1, d = 1500, 30011, 256
        h = (torch.randn(n, d, device=DEV) * hs).requires_grad_(True)
        w = (torch.randn(V1, d, device=DEV) * ws).requires_grad_(True)
        b = (torch.randn(V1, device=DEV) * 0.1).requires_grad_(True)
        labels = torch.where(torch.rand(n, device=DEV) < 0.2, torch.randint(1, V1, (n,), device=DEV), torch.zeros(n, dtype=torch.long, device=DEV))
        loss = ops.score_cross_entropy(h, labels, w, b)
        loss.backward()
        rl, rdh, rdw, rdb = _ce_ref64(h.detach(), labels, w.detach(), b.detach())
        assert abs(loss.item() - rl) < 2e-6 * abs(rl), (hs, ws, loss.item(), rl)
        for got, ref, name in ((h.grad, rdh, "dH"), (w.grad, rdw, "dW"), (b.grad, rdb, "db")):
            err = float((got.double() - ref).abs().max() / ref.abs().max())
            assert err < 1e-4, (hs, ws, name, err)


def test_score_ce_full_size_properties():
    """cfg2-sized cross-entropy (B*L = 204800 rows, 15 % scored, V + 1 = 3417, d = 64): size-independent properties -- the loss
    against an fp32 torch evaluation of the scored rows (1e-5), and sum(db) = 0, sum_v dW[v, :] = 0 (every row of
    softmax - onehot sums to zero; measured 3.4e-7 with |dW| ~ 5e-5)."""
    torch.manual_seed(11)
    n, V1, d = 204800, 3417, 64
    h = (torch.randn(n, d, device=DEV) * 0.5).requires_grad_(True)
    w = (torch.randn(V1, d, device=DEV) * 0.2).requires_grad_(True)
    b = (torch.randn(V1, device=DEV) * 0.1).requires_grad_(True)
    labels = torch.where(torch.rand(n, device=DEV) < 0.15, torch.randint(1, V1, (n,), device=DEV), torch.zeros(n, dtype=torch.long, device=DEV))
    loss = ops.score_cross_entropy(h, labels, w, b)
    loss.backward()
    sel = labels != 0
    with torch.no_grad():
        ref = F.cross_entropy(h[sel] @ w.t() + b, labels[sel])
    assert abs(loss.item() - ref.item()) < 1e-5 * abs(ref.item()), (loss.item(), ref.item())
    assert float(b.grad.sum().abs()) < 1e-5
    assert float(w.grad.sum(0).abs().max()) < 1e-5
