"""Attention kernels against float64 references whose dropout masks are computed on the host (oracle/common.py), not exported by
the library: the debug mask kernels, the dispatch of rbm_attn_fwd / rbm_attn_bwd (including the mixed layouts where one
implementation reads the stats / delta another one wrote), the live-row kernels of SASRec training and the last-query kernel of
evaluation.  Run with -m gpu on a B200; under RBM_ATTN_IMPL=mma every dense call is expected on the SIMT kernels."""
import math
import os
import re

import numpy as np
import pytest
import torch

from rbm_b200 import ops, lib as L
from oracle import common as oc

pytestmark = pytest.mark.gpu
DEV = "cuda"
MMA = os.environ.get("RBM_ATTN_IMPL") == "mma"  # the tensor-core kernels are switched off for the whole process


def attn_mask(B, h, Ln, p, seed, site, device=DEV):
    """Host-side keep mask [B, h, L, L] (bool) of an attention dropout site."""
    return torch.from_numpy(oc.attn_keep_mask(B * h, Ln, p, seed, site)).view(B, h, Ln, Ln).to(device)


def ref_attention64(q, k, v, tok, mode, scale, p, mask):
    """float64 attention on [B, h, L, dk] tensors: the reference's masked_fill(-1e9) key padding / -inf causal mask."""
    s = q @ k.transpose(-1, -2) * scale
    Ln = q.shape[-2]
    if mode == L.MASK_CAUSAL:
        s = s.masked_fill(~torch.tril(torch.ones(Ln, Ln, dtype=torch.bool, device=s.device)), float("-inf"))
    elif mode == L.MASK_KEYPAD:
        s = s.masked_fill((tok == 0)[:, None, None, :], -1e9)
    pr = torch.softmax(s, -1)
    if p > 0:
        pr = pr * mask.to(pr.dtype) / (1 - p)
    return pr @ v


def close(got, ref, rtol, atol, msg=""):
    np.testing.assert_allclose(got.detach().double().cpu().numpy(), ref.detach().double().cpu().numpy(), rtol=rtol, atol=atol, err_msg=msg)


def heads(x, B, Ln, h):
    return x.view(B, Ln, h, -1).transpose(1, 2)


def unheads(x):
    B, h, Ln, dk = x.shape
    return x.transpose(1, 2).reshape(B * Ln, h * dk)


# ------------------------------------------------------------------------------------------------ dropout masks (§ host oracle)
@pytest.mark.parametrize("Ln", [1, 7, 16, 17, 64, 200, 256])
@pytest.mark.parametrize("p", [0.1, 0.3, 0.5, 0.77777])
def test_dropout_masks_bit_equal_to_host(Ln, p):
    """rbm_dropout_mask / rbm_dropout_mask_attn equal the host restatement bit for bit: seeds with the high 32 bits set, sites
    >= 2^32, thresholds that round up (p * 65536 = 6553.6, 19660.8, 50972.4)."""
    for seed, site in ((5, 11), ((0xDEADBEEF << 32) | 123, (7 << 32) | 64 * 1000 + 3)):
        BH = 5
        got = ops.dropout_mask_attn(BH * Ln, Ln, p, seed, site, DEV).cpu().numpy().astype(bool)
        np.testing.assert_array_equal(got, oc.attn_keep_mask(BH, Ln, p, seed, site))
        n = BH * Ln * 16 + 3  # ragged tail of the last Philox call
        got = ops.dropout_mask(n, p, seed, site, DEV).cpu().numpy().astype(bool)
        np.testing.assert_array_equal(got, oc.keep_mask(n, p, seed, site))


def test_attn_mask_call_index_past_2_32():
    """L = 1 with B*h > 2^19 sequence-heads: the Philox call index bh * 8192 crosses 2^32 (its high word becomes non-zero)."""
    BH, p, seed, site = (1 << 19) + 1000, 0.25, (3 << 40) | 9, 1 << 33
    got = ops.dropout_mask_attn(BH, 1, p, seed, site, DEV).cpu().numpy().astype(bool)
    ref = oc.attn_keep_mask(BH, 1, p, seed, site)
    np.testing.assert_array_equal(got, ref)
    assert 0.7 < ref[1 << 19:].mean() < 0.8  # the rows past the crossing are not all one value


# -------------------------------------------------------------------------------------- direct calls of rbm_attn_fwd / _bwd
def _fwd(q, k, v, tok, out, ldo, stats, B, Ln, h, dk, mode, scale, p, seed, site):
    lib = L.load()
    L.check(lib.rbm_attn_fwd(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), L.ptr(tok), out, ldo,
                             stats.data_ptr(), B, Ln, h, dk, mode, scale, p, seed, site, L.stream()), "attn_fwd")


def _bwd(q, k, v, tok, out, ldo, dout, stats, dq, dk_, dv, ld, B, Ln, h, dk, mode, scale, p, seed, site):
    """dq / dk_ / dv are raw device addresses with row stride ``ld``."""
    lib = L.load()
    nb = lib.rbm_attn_bwd_ws_bytes(B, Ln, h)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    L.check(lib.rbm_attn_bwd(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0), L.ptr(tok), out, ldo,
                             dout.data_ptr(), dout.stride(0), stats.data_ptr(), dq, ld, dk_, ld, dv, ld, B, Ln, h, dk, mode, scale, p,
                             seed, site, ws.data_ptr(), nb, L.stream()), "attn_bwd")


def _inputs(B, Ln, h, dk, seed):
    torch.manual_seed(seed)
    d = h * dk
    q, k, v, dout = (torch.randn(B * Ln, d, device=DEV) for _ in range(4))
    tok = torch.randint(1, 50, (B, Ln), device=DEV)
    tok[0, : Ln // 3] = 0
    if B > 1:
        tok[1, :] = 0
    return q, k, v, dout, tok


def _misaligned(rows, cols):
    """[rows, cols] fp32 view whose base address is 8-byte but not 16-byte aligned, and its storage."""
    buf = torch.empty(rows * cols + 4, device=DEV)
    assert buf.data_ptr() % 16 == 0
    return buf[2: 2 + rows * cols].view(rows, cols), buf


def _run_layout(layout, B, Ln, h, dk, mode, p, seed=3, site=17):
    """One forward + backward through the C ABI with ``out`` (layout "out8") or dk / dv (layout "dkv8") 8-byte aligned;
    returns (out, dq, dk, dv, inputs)."""
    q, k, v, dout, tok = _inputs(B, Ln, h, dk, 11)
    d = h * dk
    scale = 1 / math.sqrt(dk)
    if layout == "out8":
        out, _keep = _misaligned(B * Ln, d)
    else:
        out = torch.empty(B * Ln, d, device=DEV)
    stats = torch.empty(B * h * Ln, 2, device=DEV)
    _fwd(q, k, v, tok, out.data_ptr(), d, stats, B, Ln, h, dk, mode, scale, p, seed, site)
    dq = torch.empty(B * Ln, d, device=DEV)
    if layout == "dkv8":
        dkb, _k1 = _misaligned(B * Ln, d)
        dvb, _k2 = _misaligned(B * Ln, d)
    else:
        dkb, dvb = torch.empty(B * Ln, d, device=DEV), torch.empty(B * Ln, d, device=DEV)
    ld = d
    _bwd(q, k, v, tok, out.data_ptr(), d, dout, stats, dq.data_ptr(), dkb.data_ptr(), dvb.data_ptr(), ld, B, Ln, h, dk, mode, scale, p,
         seed, site)
    torch.cuda.synchronize()
    return out.clone(), dq, dkb.clone(), dvb.clone(), (q, k, v, dout, tok, scale, seed, site)


def _ref_grads(q, k, v, dout, tok, B, Ln, h, mode, scale, p, seed, site):
    qd, kd, vd = (heads(x.double(), B, Ln, h).detach().requires_grad_(True) for x in (q, k, v))
    mask = attn_mask(B, h, Ln, p, seed, site) if p > 0 else None
    o = ref_attention64(qd, kd, vd, tok, mode, scale, p, mask)
    o.backward(heads(dout.double(), B, Ln, h))
    return unheads(o), unheads(qd.grad), unheads(kd.grad), unheads(vd.grad)


@pytest.mark.skipif(MMA, reason="the mixed layouts mix the tensor-core and SIMT kernels")
@pytest.mark.parametrize("layout", ["out8", "dkv8"])
@pytest.mark.parametrize("mode", [L.MASK_NONE, L.MASK_CAUSAL, L.MASK_KEYPAD])
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_attention_mixed_layouts(layout, mode, p):
    """d_k = 32 with an 8-byte aligned output (SIMT forward and dQ, tcgen05 dK/dV) or 8-byte aligned dK/dV (tcgen05 forward and dQ,
    SIMT dK/dV): the kernels of one family consume the stats / delta written by the other."""
    B, Ln, h, dk = 4, 77, 2, 32
    out, dq, dk_, dv, (q, k, v, dout, tok, scale, seed, site) = _run_layout(layout, B, Ln, h, dk, mode, p)
    ro, rq, rk, rv = _ref_grads(q, k, v, dout, tok, B, Ln, h, mode, scale, p, seed, site)
    close(out, ro, 1e-4, 1e-5, "out")
    close(dq, rq, 1e-3, 2e-5, "dq")
    close(dk_, rk, 1e-3, 2e-5, "dk")
    close(dv, rv, 1e-3, 2e-5, "dv")


# ------------------------------------------------------------------------------------------------------------ dispatch
_SIMT = ("attn_fwd_kernel", "attn_bwd_dq_kernel", "attn_bwd_dkv_kernel")
_TC = ("attn_fwd_tc_kernel", "attn_bwd_dq_tc_kernel", "attn_bwd_dkv_tc_kernel")
_PAIR = ("attn_pair_fwd_kernel", "attn_pair_bwd_kernel")
_SEQ = ("attn_seq_fwd_kernel", "attn_seq_dq_kernel", "attn_seq_dkv_kernel")
_ALL = _SIMT + _TC + _PAIR + _SEQ
# (name, layout, B, L, h, d_k, mask) -> kernels expected with the tensor paths on
DISPATCH = [
    ("tc_dk32", "plain", 3, 50, 2, 32, L.MASK_CAUSAL, _TC),
    ("pair_dk64_L<=64", "plain", 3, 50, 1, 64, L.MASK_CAUSAL, _PAIR),
    ("seq_dk64_64<L<=256", "plain", 2, 129, 1, 64, L.MASK_KEYPAD, _SEQ),
    ("simt_dk16", "plain", 2, 40, 2, 16, L.MASK_CAUSAL, _SIMT),
    ("simt_dk64_keypad_L<=64", "plain", 2, 40, 1, 64, L.MASK_KEYPAD, _SIMT),
    ("mixed_out8", "out8", 2, 40, 2, 32, L.MASK_CAUSAL, ("attn_fwd_kernel", "attn_bwd_dq_kernel", "attn_bwd_dkv_tc_kernel")),
    ("mixed_dkv8", "dkv8", 2, 40, 2, 32, L.MASK_CAUSAL, ("attn_fwd_tc_kernel", "attn_bwd_dq_tc_kernel", "attn_bwd_dkv_kernel")),
]


def _kernel_names():
    from torch.profiler import profile, ProfilerActivity
    return profile(activities=[ProfilerActivity.CUDA])


def _ran(names, kernel):
    """Whether a kernel of that exact name (demangled `ns::name<...>(` or mangled `<len>name<I|E>`) is among the launches."""
    pat = re.compile(r"(?<![A-Za-z_])%s(?![a-z_])" % kernel)
    return any(pat.search(n) for n in names)


@pytest.mark.parametrize("row", DISPATCH, ids=[r[0] for r in DISPATCH])
def test_attention_dispatch_reaches_every_path(row):
    """Each row of the rbm_attn_fwd / rbm_attn_bwd dispatch runs the kernels it is meant to (and none of another path): a change
    of a dispatch condition names the path that no longer runs.  Under RBM_ATTN_IMPL=mma every row runs the SIMT kernels."""
    name, layout, B, Ln, h, dk, mode, expect = row
    if MMA:
        expect = _SIMT
    with _kernel_names() as prof:
        _run_layout("plain" if layout == "plain" else layout, B, Ln, h, dk, mode, 0.1)
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    for kern in expect:
        assert _ran(names, kern), (name, kern, sorted(set(names)))
    for kern in _ALL:
        if kern not in expect:
            assert not _ran(names, kern), (name, kern, sorted(set(names)))


# ----------------------------------------------------------------------------------- split-fp16 paths: dynamic range of dO
@pytest.mark.skipif(MMA, reason="the split-fp16 kernels are switched off")
@pytest.mark.parametrize("Ln", [64, 200])
def test_attention_split_fp16_dout_range(Ln):
    """pair (L <= 64) and seq (64 < L <= 256) kernels keep fp16 hi / lo halves scaled per tile by a power of two: dO rows spanning
    10^-3 .. 10^3 inside one (sequence, head) tile.  The promise is accuracy relative to the tile's largest value; the per-row
    relative error is printed (pytest -s)."""
    B, h, dk, mode, p = 3, 2, 64, L.MASK_CAUSAL, 0.1
    q, k, v, dout, tok = _inputs(B, Ln, h, dk, 5)
    dout = dout * (10.0 ** torch.linspace(-3, 3, B * Ln, device=DEV)[torch.randperm(B * Ln, device=DEV)])[:, None]
    d = h * dk
    scale = 1 / math.sqrt(dk)
    qkv = torch.cat([q, k, v], 1).requires_grad_(True)
    out = ops.attention(qkv, None, tok, B, Ln, h, 0, d, 2 * d, mode, scale, p, 3, 17)
    out.backward(dout)
    _, rq, rk, rv = _ref_grads(q, k, v, dout, tok, B, Ln, h, mode, scale, p, 3, 17)
    g = qkv.grad
    for got, ref, nm in ((g[:, :d], rq, "dq"), (g[:, d:2 * d], rk, "dk"), (g[:, 2 * d:], rv, "dv")):
        e = heads((got.double() - ref).abs(), B, Ln, h)
        r = heads(ref.abs(), B, Ln, h)
        tile_err = (e.amax((2, 3)) / r.amax((2, 3))).max().item()
        rmax = r.amax(3)
        live = rmax > 1e-12 * r.amax((2, 3), keepdim=True)[..., 0]  # rows whose exact value is 0 (a lone key: P = 1) have no relative error
        row_err = (e.amax(3)[live] / rmax[live]).max().item()
        print("L=%d %s: max error / tile max %.3g, max per-row relative error %.3g" % (Ln, nm, tile_err, row_err))
        assert tile_err < 1e-4, (nm, tile_err)


# ---------------------------------------------------------------------------------------------- live-row attention (SASRec)
def _live_tokens(B, Ln, gen):
    """[B, L] token ids: left-padded histories of random length plus the edge patterns (empty, fully live, interior padding,
    only the last position live); position L-1 of every non-empty left-padded sequence is live (position 63 at L = 64)."""
    tok = torch.zeros(B, Ln, dtype=torch.long)
    for b in range(B):
        kind = b % 6
        if kind == 1:
            continue  # empty sequence
        row = torch.randint(1, 1000, (Ln,), generator=gen)
        if kind == 0:
            n = int(torch.randint(1, Ln + 1, (1,), generator=gen))
            row[: Ln - n] = 0  # left padding (Amazon-Beauty-like)
        elif kind == 3:
            row[torch.rand(Ln, generator=gen) < 0.4] = 0  # padding inside the sequence
        elif kind == 4:
            row[:-1] = 0  # only the last position
        elif kind == 5 and Ln > 2:
            row[Ln // 2] = 0  # one dead key in the middle, live keys on both sides
        tok[b] = row
    return tok


def _live_call(B, Ln, h, dk, p, extra, seed=21, site=5 + (1 << 34), gseed=0):
    """Compact inputs (NaN in rows past the count), the live kernels' outputs (sentinels outside the written rows) and the tensors
    needed to rebuild the dense reference."""
    gen = torch.Generator().manual_seed(gseed + 1000 * Ln + 10 * dk + h)
    tok = _live_tokens(B, Ln, gen).to(DEV)
    n_live = int((tok != 0).sum())
    cap = n_live + extra
    live = ops.LiveRows(tok, cap)
    d = h * dk
    q = torch.full((cap, d), float("nan"), device=DEV)
    kv = torch.full((cap, 2 * d), float("nan"), device=DEV)
    dout = torch.full((cap, d), float("nan"), device=DEV)
    q[:n_live] = torch.randn(n_live, d, generator=gen).to(DEV)
    kv[:n_live] = torch.randn(n_live, 2 * d, generator=gen).to(DEV)
    dout[:n_live] = torch.randn(n_live, d, generator=gen).to(DEV)
    bkv = torch.randn(2 * d, generator=gen).to(DEV)
    SENT = -12345.0
    out = torch.full((cap, d), SENT, device=DEV)
    stats = torch.full((cap, h, 2), SENT, device=DEV)
    dq = torch.full((cap, d), SENT, device=DEV)
    dkv = torch.full((cap, 2 * d), SENT, device=DEV)
    dead = torch.full((cap, 2 * d), SENT, device=DEV)
    delta = torch.empty(cap, h, device=DEV)
    keepw = torch.empty(cap, h, dtype=torch.int64, device=DEV)
    scale = 1 / math.sqrt(dk)
    lib = L.load()
    P = L.ptr
    L.check(lib.rbm_attn_live_fwd(P(q), d, P(kv), 2 * d, P(bkv), P(live.rows), P(live.seq_start), P(live.tok), P(out), P(stats), B, Ln, h,
                                  dk, scale, p, seed, site, L.stream()), "attn_live_fwd")
    L.check(lib.rbm_attn_live_bwd(P(q), d, P(kv), 2 * d, P(bkv), P(live.rows), P(live.seq_start), P(live.tok), P(out), P(stats), P(dout),
                                  P(dq), P(dkv), P(dead), P(delta), P(keepw), B, Ln, h, dk, scale, p, seed, site, L.stream()),
            "attn_live_bwd")
    dbkv = torch.full((2 * d,), SENT, device=DEV)
    nb = lib.rbm_rows_dead_colsum_ws_bytes(2 * d)
    ws = torch.empty(nb, dtype=torch.uint8, device=DEV)
    L.check(lib.rbm_rows_live_colsum(P(dead), 2 * d, P(live.count), cap, 2 * d, P(dbkv), P(ws), nb, L.stream()), "rows_live_colsum")
    torch.cuda.synchronize()
    assert int(live.count) == n_live
    return dict(tok=tok, n=n_live, cap=cap, q=q, kv=kv, dout=dout, bkv=bkv, out=out, stats=stats, dq=dq, dkv=dkv, dead=dead, dbkv=dbkv,
                scale=scale, seed=seed, site=site, SENT=SENT)


def _live_reference(r, B, Ln, h, dk, p):
    """Dense causal attention on the [B, L] layout in float64: live rows from the compact tensors, every padding key / value = bkv."""
    n, d = r["n"], h * dk
    live = (r["tok"] != 0).reshape(-1)
    qc = r["q"][:n].double().requires_grad_(True)
    kvc = r["kv"][:n].double().requires_grad_(True)
    bkv = r["bkv"].double().requires_grad_(True)
    Q = torch.zeros(B * Ln, d, dtype=torch.float64, device=DEV).index_put((live.nonzero()[:, 0],), qc)
    KV = bkv.expand(B * Ln, 2 * d).index_put((live.nonzero()[:, 0],), kvc)
    mask = attn_mask(B, h, Ln, p, r["seed"], r["site"]) if p > 0 else None
    qh, kh, vh = heads(Q, B, Ln, h), heads(KV[:, :d], B, Ln, h), heads(KV[:, d:], B, Ln, h)
    s = qh @ kh.transpose(-1, -2) * r["scale"]
    s = s.masked_fill(~torch.tril(torch.ones(Ln, Ln, dtype=torch.bool, device=DEV)), float("-inf"))
    mx = s.amax(-1)
    pr = torch.softmax(s, -1)
    inv = 1.0 / torch.exp(s - mx[..., None]).sum(-1)
    if p > 0:
        pr = pr * mask.double() / (1 - p)
    o = unheads(pr @ vh)[live]
    o.backward(r["dout"][:n].double())
    stats = torch.stack([mx, inv], -1).transpose(1, 2).reshape(B * Ln, h, 2)[live]
    return o.detach(), stats.detach(), qc.grad, kvc.grad, bkv.grad


def _check_live(r, B, Ln, h, dk, p):
    n, cap, SENT = r["n"], r["cap"], r["SENT"]
    o, st, gq, gkv, gb = _live_reference(r, B, Ln, h, dk, p)
    close(r["out"][:n], o, 1e-4, 1e-5, "out")
    close(r["stats"][:n], st, 1e-4, 1e-5, "stats")
    close(r["dq"][:n], gq, 1e-3, 2e-5, "dq")
    close(r["dkv"][:n], gkv, 1e-3, 2e-5, "dkv")
    close(r["dbkv"], gb, 1e-3, 2e-5 * max(1.0, math.sqrt(n / 100)), "dbkv")  # a column sum over n rows
    for nm in ("out", "stats", "dq", "dkv", "dead"):
        assert not torch.isnan(r[nm][:n]).any(), nm
        assert bool((r[nm][n:cap] == SENT).all()), "%s: rows past the count were written" % nm


@pytest.mark.parametrize("dk", [16, 32, 64, 128])
@pytest.mark.parametrize("h", [1, 2, 3])
@pytest.mark.parametrize("Ln", [1, 4, 5, 50, 63, 64])
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_attention_live_rows(dk, h, Ln, p):
    """rbm_attn_live_fwd / _bwd + rbm_rows_live_colsum against float64 dense causal attention: out, stats (row maximum and 1 / row
    sum in natural units), dq, dkv, d bkv; rows past the count hold NaN inputs and must stay unwritten."""
    B = 14
    r = _live_call(B, Ln, h, dk, p, extra=5)
    _check_live(r, B, Ln, h, dk, p)


@pytest.mark.parametrize("B,Ln,h,dk", [(4096, 50, 2, 64), (600, 64, 3, 16)])
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_attention_live_rows_grid_stride(B, Ln, h, dk, p):
    """More warp items (B * h * ceil(L / 4) = 106,496 at the SASRec bench shape, 28,800) than the capped grid's 7,104 warps:
    every warp walks several items."""
    r = _live_call(B, Ln, h, dk, p, extra=37)
    _check_live(r, B, Ln, h, dk, p)


@pytest.mark.parametrize("Ln,dk,h", [(50, 64, 2), (64, 32, 1), (5, 128, 3)])
@pytest.mark.parametrize("p", [0.0, 0.2])
def test_attention_live_matches_dense_kernels(Ln, dk, h, p):
    """The same inputs through rbm_attn_fwd / rbm_attn_bwd on the scattered [B, L] layout (padding rows: zero queries, bkv as key /
    value -- what models/sas.py does for L > 64) agree with the live-row kernels."""
    B = 30
    r = _live_call(B, Ln, h, dk, p, extra=0)
    n, d = r["n"], h * dk
    live = ops.LiveRows(r["tok"], n)
    q = ops.rows_scatter(r["q"], None, live).requires_grad_(True)
    kv = ops.rows_scatter(r["kv"], r["bkv"], live).requires_grad_(True)
    ctx = ops.attention(q, kv, None, B, Ln, h, 0, 0, d, L.MASK_CAUSAL, r["scale"], p, r["seed"], r["site"])
    ctx_c = ops.rows_gather(ctx.view(-1, d), live)
    ctx_c.backward(r["dout"])
    livem = (r["tok"] != 0).reshape(-1)
    close(r["out"][:n], ctx_c[:n], 1e-4, 1e-5, "out")
    close(r["dq"][:n], q.grad[livem], 1e-3, 2e-5, "dq")
    close(r["dkv"][:n], kv.grad[livem], 1e-3, 2e-5, "dkv")
    close(r["dbkv"], kv.grad[~livem].sum(0), 1e-3, 1e-4, "dbkv")


# --------------------------------------------------------------------------------------------------- last-query attention
@pytest.mark.parametrize("dk", [4, 16, 32, 64, 128])
@pytest.mark.parametrize("Ln", [1, 50, 128, 129, 200, 256])
@pytest.mark.parametrize("mode", [L.MASK_NONE, L.MASK_CAUSAL, L.MASK_KEYPAD])
@pytest.mark.parametrize("packed", [2, 3])
def test_attention_last_query(dk, Ln, mode, packed):
    """rbm_attn_last_query against the last row of float64 full attention and of rbm_attn_fwd (d_k >= 8): k / v are column slices
    of a packed [B*L, packed*d] tensor (ld = 2d with k | v, ld = 3d with q | k | v); key padding with a fully padded sequence."""
    B, h = 5, 2
    d = h * dk
    torch.manual_seed(Ln * dk + mode)
    big = torch.randn(B * Ln, packed * d, device=DEV)
    kc, vc = (packed - 2) * d, (packed - 1) * d
    qfull = torch.randn(B * Ln, d, device=DEV)
    q = qfull.view(B, Ln, d)[:, -1, :].contiguous()
    tok = torch.randint(1, 50, (B, Ln), device=DEV)
    tok[0, : Ln // 3] = 0
    tok[1, :] = 0
    tok[2, :-1] = 0
    scale = 1 / math.sqrt(dk)
    with torch.no_grad():
        out = ops.attention_last_query(q, big, tok if mode == L.MASK_KEYPAD else None, B, Ln, h, kc, vc, mode, scale)
        kh, vh = heads(big[:, kc:kc + d].double(), B, Ln, h), heads(big[:, vc:vc + d].double(), B, Ln, h)
        qh = heads(qfull.double(), B, Ln, h)
        ref = unheads(ref_attention64(qh, kh, vh, tok, mode, scale, 0.0, None)).view(B, Ln, d)[:, -1, :]
        close(out, ref, 1e-4, 1e-5, "vs float64")
        if dk >= 8:
            try:
                full = ops.attention(qfull, big, tok, B, Ln, h, 0, kc, vc, mode, scale).view(B, Ln, d)[:, -1, :]
            except RuntimeError as e:  # the SIMT kernel's K / V panels of d_k = 128 at L >= 200 do not fit shared memory
                assert "unsupported shape" in str(e) and dk == 128, e
                return
            close(out, full, 1e-4, 1e-5, "vs rbm_attn_fwd")


def test_attention_last_query_empty_batch():
    """B = 0 is a valid call: it returns 0 and writes nothing."""
    lib = L.load()
    q, kv = torch.randn(4, 64, device=DEV), torch.randn(4 * 8, 128, device=DEV)
    out = torch.full((4, 64), 3.0, device=DEV)
    rc = lib.rbm_attn_last_query(q.data_ptr(), 64, kv.data_ptr(), 128, kv.data_ptr() + 4 * 64, 128, None, out.data_ptr(), 64, 0, 8, 2,
                                 32, L.MASK_CAUSAL, 0.1, L.stream())
    torch.cuda.synchronize()
    assert rc == 0
    assert bool((out == 3.0).all())
