"""Row-wise kernels against float64: LayerNorm (csrc/layernorm.cu), the embedding stage (csrc/embed.cu), the live-row layouts
(csrc/rows.cu, rbm_rows_seq_start), SASRec scoring, BCE and candidate scores (csrc/sas_score.cu), the metric column mean, Adam and
the gradient-bucket pack (csrc/adam.cu).  Every kernel is called through the C ABI so that each output is checked on its own.
Every reference takes the fp32 inputs the kernel saw, promoted to float64; dropout masks come from the host Philox
(oracle.common.keep_mask).  Run with -m gpu on a B200; `pytest -s` prints the largest error / bar per family.

Error model.  u = 2^-24 (fp32 unit roundoff).  A sum whose additions form a tree of depth D is off by at most D * u * (sum of the
magnitudes of its terms); every bar below is that, with D read off the kernel's summation order, plus a few u per element-wise
operation.  These are worst-case bounds.  Largest error / bar measured on a B200 (1000 W power limit): LayerNorm 0.11, large-mean
LayerNorm 0.11 of its torch-relative bar, embedding 0.67, live-row embedding 0.52, column sums 0.11, SASRec scoring 0.96 (df, whose
2 u bound is exact for its two roundings), BCE 0.43, candidate scores 0.15, column mean 0.5 ulp, Adam 0.40.

  * LayerNorm, per row with rstd r, mean |x| = mx, |xhat| + r * mx = xs (xhat's magnitude plus the error scale of the fp32 mean),
    A = |dy| + |dy2|, gA = A |gamma|, C = 32 >= the depth of the row sums (3 NV + log2 GW <= 29) plus the element-wise roundings:
      mean: C u mx;  rstd: C u r (1 + C u (r mx)^2);  y: C u (|gamma| xs + |beta|);
      dx: C u (r (gA + mean gA) + r xs mean(gA xs) [* d/(d-1) for BERT] + |dres|);
      dbeta: (D + 2) u sum_rows A;  dgamma: (D + C + 2) u sum_rows A xs,
    with D = ceil(rows_per_block / row groups) + row groups + ceil(blocks / 32) + 32 (ln_bwd_blocks and colsum_partials_kernel).
    A dropped dres or dy2 changes dx by |dres| or r |gamma dy2| = O(1), against a bar of O(1e-5).
    Rows with mean 1e3 and spread 1e-2 lose about r * mx * u = 1e5 u in any fp32 implementation; there each quantity's largest
    error must stay within 8 x that of torch's fp32 LayerNorm (CPU, same fp64 reference) + 2^-20 max |ref|.
  * Embedding forward: 3 u (|table * scale| + |pos|) / (1 - p) (one fused multiply-add, the dropout scale, its fp32 rounding).
    g: 2 u |g|.  dpos = column sums over the batch: (D + 2) u sum |g|, D = ceil(B / 16) + 16 (+ the number of rank slices when
    their results are added); live-row kernel D = ceil(count / 148) + 148.  Table gradient (sorted scatter): (n_v + 3) u sum |terms|
    over the n_v contributions of row v.  Shard sums, slices of the global backward and the live-row g are bit-exact.
  * Row moves (rows_to_seq, seq_to_rows, rows_gather) are bit-exact; dead / live column sums (D + 2) u sum |x| with
    D = ceil(per / row lanes) + row lanes + ceil(1184 / 256) + 8, per = ceil(n / 1184), row lanes = 256 / (d / 4).
  * SASRec logits and candidate scores: (ceil(d/4 / gw) + log2 gw + 4) u (sum |f t| + |bias|); df: 2 u (|dpl t_p| + |dnl t_n|).
  * BCE loss: (D + 8) u (sum softplus) / count, D = 4 + 8 + ceil(rows / 1024); dpl: 8 u |g| (s + |1 - s|) + 2^-126 |g|, dnl:
    8 u |g| s + 2^-126 |g| (s = sigmoid, g = dloss / count; 2^-126 covers the sigmoid that fp32 flushes to 0 or 1).
  * Column mean (double accumulation): 1 fp32 ulp of the exact mean.
  * Adam: a first-order error bound propagated alongside the fp64 trajectory (oracle.optim.adam_step run on float64 arrays with the
    same fp32 hyper-parameters), one rounding per operation, doubled (_adam_bound).
  * Bit-exact: run-to-run repeats of every fixed-order reduction, device step counter vs eager step, bucket pack / unpack with a
    power-of-two scale.

A skipped partial block in a column sum would be off by that block's contribution: the column-sum tests assert, per non-empty
block, that this contribution exceeds the bar in some column (_each_block_matters), so no bar can hide a missing block.  An
off-by-one row_offset reorders the dropout stream and breaks the bit-exact slice check.
"""
import math
from collections import defaultdict

import numpy as np
import pytest
import torch

from rbm_b200 import dist as rd, ops, lib as L
from oracle import common as oc, optim as oo

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)
U = 2.0 ** -24
NSM = 148
NAN = float("nan")
SEED, SITE = 0x5EED1234, 77
WORST = defaultdict(float)  # family -> largest error / bar


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nlargest error / bar per family (bit-exact checks not listed)")
    for k in sorted(WORST):
        print("  %-34s %.3g" % (k, WORST[k]))


def lib():
    return L.load()


P, S = L.ptr, L.stream


def _check(fam, got, ref, bar, what=""):
    """|got - ref| <= bar element-wise (ref, bar float64); records the largest ratio for the family."""
    got = got.double()
    assert not bool(torch.isnan(got).any()), (fam, what, "NaN in output")
    err = (got - ref).abs()
    r = torch.where(err == 0, torch.zeros_like(err), err / bar)
    r = float(r.max()) if r.numel() else 0.0
    WORST[fam] = max(WORST[fam], r)
    assert r <= 1.0, (fam, what, r)


def _each_block_matters(contrib, bar, what):
    """contrib [blocks, ...] float64 = what each partial block adds to the column sums: each non-empty block must move some column
    by more than its bar, so a kernel that skipped it would fail the comparison."""
    c = contrib.reshape(contrib.shape[0], -1).abs()
    nonempty = c.sum(1) > 0
    seen = (c > bar.reshape(1, -1)).any(1)
    assert bool((seen | ~nonempty).all()), (what, "a block's share is within the bar", int((~seen & nonempty).sum()))


def _gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def _mask64(n, p):
    """Dropout factor per element in float64: keep / (1 - p), p rounded to fp32 as the C ABI passes it."""
    keep = torch.from_numpy(oc.keep_mask(n, p, SEED, SITE)).to(DEV)
    return keep.double() / (1.0 - float(np.float32(p)))


# ================================================================================================================ LayerNorm
LN_EPS = {L.LN_TORCH: 1e-8, L.LN_BERT: 1e-6}
C_LN = 32


def ln_partition(rows, d):
    """(blocks, rows per block, depth D of the dgamma / dbeta sums) as ln_bwd_blocks and the kernels lay them out."""
    nblk = min(max(-(-rows // 128), 1), 4 * NSM)
    rpb = -(-rows // nblk)
    d4 = d // 4
    ng = 256 // (8 if d4 <= 8 else 16 if d4 <= 16 else 32)
    return nblk, rpb, -(-rpb // ng) + ng + -(-nblk // 32) + 32


def ln_fwd(x, gamma, beta, flavour):
    rows, d = x.shape
    y = torch.full_like(x, NAN)
    stats = torch.full((rows, 2), NAN, device=DEV)
    L.check(lib().rbm_layernorm_fwd(P(x), P(gamma), P(beta), P(y), P(stats), rows, d, LN_EPS[flavour], flavour, S()), "ln_fwd")
    return y, stats


def ln_bwd(entry, x, gamma, dy, dy2, dres, stats, flavour, ws=None):
    """One backward through `entry` on a workspace and outputs filled with NaN first (every value must be overwritten)."""
    rows, d = x.shape
    nb = lib().rbm_layernorm_ws_bytes(rows, d)
    if ws is None:
        ws = torch.full((nb // 4,), NAN, device=DEV)
    dx, dg, db = torch.full_like(x, NAN), torch.full((d,), NAN, device=DEV), torch.full((d,), NAN, device=DEV)
    eps = LN_EPS[flavour]
    if entry == "bwd":
        assert dy2 is None and dres is None
        rc = lib().rbm_layernorm_bwd(P(x), P(gamma), P(dy), P(stats), P(dx), P(dg), P(db), rows, d, eps, flavour, P(ws), nb, S())
    elif entry == "residual":
        assert dy2 is None
        rc = lib().rbm_layernorm_bwd_residual(P(x), P(gamma), P(dy), P(dres), P(stats), P(dx), P(dg), P(db), rows, d, eps, flavour,
                                              P(ws), nb, S())
    else:
        rc = lib().rbm_layernorm_bwd_fanout(P(x), P(gamma), P(dy), P(dy2), P(dres), P(stats), P(dx), P(dg), P(db), rows, d, eps,
                                            flavour, P(ws), nb, S())
    L.check(rc, entry)
    return dx, dg, db


def ln_ref64(x, gamma, beta, flavour, G=None, dres=None):
    """LN(x) in float64 and, for an upstream gradient G (= dy + dy2), the gradients; dx includes dres."""
    d = x.shape[1]
    eps = float(np.float32(LN_EPS[flavour]))
    need = G is not None
    xx, gg, bb = (t.double().requires_grad_(need) for t in (x, gamma, beta))
    mu = xx.mean(1, keepdim=True)
    xc = xx - mu
    if flavour == L.LN_TORCH:
        r = torch.rsqrt((xc * xc).mean(1, keepdim=True) + eps)
    else:
        r = 1.0 / (torch.sqrt((xc * xc).sum(1, keepdim=True) / (d - 1)) + eps)
    y = xc * r * gg + bb
    out = {"y": y.detach(), "mean": mu.detach()[:, 0], "rstd": r.detach()[:, 0]}
    if need:
        y.backward(G)
        out["dx"] = xx.grad + (0.0 if dres is None else dres.double())
        out["dgamma"], out["dbeta"] = gg.grad, bb.grad
    return out


def ln_bars(x, gamma, beta, ref, flavour, dy=None, dy2=None, dres=None, depth=0):
    d = x.shape[1]
    x64, r = x.double(), ref["rstd"][:, None]
    mx = x64.abs().mean(1, keepdim=True)
    xs = (x64 - ref["mean"][:, None]).abs() * r + r * mx
    ga = gamma.double().abs()
    bars = {"mean": C_LN * U * mx[:, 0], "rstd": C_LN * U * ref["rstd"] * (1 + C_LN * U * (r * mx)[:, 0] ** 2),
            "y": C_LN * U * (ga * xs + beta.double().abs())}
    if dy is not None:
        A = dy.double().abs() + (0.0 if dy2 is None else dy2.double().abs())
        gA = A * ga
        f = d / (d - 1) if flavour == L.LN_BERT else 1.0
        bars["dx"] = C_LN * U * (r * (gA + gA.mean(1, keepdim=True)) + r * xs * (gA * xs).mean(1, keepdim=True) * f
                                 + (0.0 if dres is None else dres.double().abs()))
        bars["dbeta"] = (depth + 2) * U * A.sum(0)
        bars["dgamma"] = (depth + C_LN + 2) * U * (A * xs).sum(0)
    return bars


def ln_inputs(rows, d, seed, xscale=2.0, xshift=0.5):
    g = _gen(seed)
    x = torch.randn(rows, d, device=DEV, generator=g) * xscale + xshift
    gamma, beta = torch.randn(d, device=DEV, generator=g), torch.randn(d, device=DEV, generator=g)
    dy, dy2, dres = (torch.randn(rows, d, device=DEV, generator=g) for _ in range(3))
    return x, gamma, beta, dy, dy2, dres


def ln_check_fwd(fam, x, gamma, beta, flavour, what):
    y, stats = ln_fwd(x, gamma, beta, flavour)
    ref = ln_ref64(x, gamma, beta, flavour)
    bars = ln_bars(x, gamma, beta, ref, flavour)
    _check(fam, y, ref["y"], bars["y"], what + " y")
    _check(fam, stats[:, 0], ref["mean"], bars["mean"], what + " mean")
    _check(fam, stats[:, 1], ref["rstd"], bars["rstd"], what + " rstd")
    return stats


def ln_check_bwd(fam, entry, x, gamma, beta, dy, dy2, dres, stats, flavour, what):
    dx, dg, db = ln_bwd(entry, x, gamma, dy, dy2, dres, stats, flavour)
    G = dy.double() + (0.0 if dy2 is None else dy2.double())
    ref = ln_ref64(x, gamma, beta, flavour, G, dres)
    bars = ln_bars(x, gamma, beta, ref, flavour, dy, dy2, dres, ln_partition(*x.shape)[2])
    for nm, got in (("dx", dx), ("dgamma", dg), ("dbeta", db)):
        _check(fam, got, ref[nm], bars[nm], "%s %s %s" % (what, entry, nm))
    return (dx, dg, db), ref, bars


# (entry point, with dy2, with dres)
LN_VARIANTS = [("bwd", False, False), ("residual", False, True), ("residual", False, False), ("fanout", True, True),
               ("fanout", True, False), ("fanout", False, True), ("fanout", False, False)]
# every (NV, GW) bucket of the forward and backward, each with a width that leaves lanes idle; 772 and 1024 take the opt-in
# shared memory of the backward (8 row groups x 2 x d floats > 48 KB)
LN_WIDTHS = [4, 12, 32, 36, 64, 68, 128, 132, 256, 260, 516, 772, 1024]


@pytest.mark.parametrize("d", LN_WIDTHS)
@pytest.mark.parametrize("flavour", [L.LN_TORCH, L.LN_BERT], ids=["torch", "bert"])
def test_layernorm_widths(flavour, d):
    """y, mean and rstd of the forward; dx, dgamma and dbeta of rbm_layernorm_bwd, _bwd_residual (with and without dres) and
    _bwd_fanout (every combination of dy2 and dres) against the float64 gradient of LN(x) with upstream dy + dy2, plus dres.
    At d = 4 the BERT flavour divides by d - 1 = 3."""
    x, gamma, beta, dy, dy2, dres = ln_inputs(300, d, seed=d * 7 + flavour)
    stats = ln_check_fwd("layernorm", x, gamma, beta, flavour, "d=%d" % d)
    for entry, w2, wr in LN_VARIANTS:
        ln_check_bwd("layernorm", entry, x, gamma, beta, dy, dy2 if w2 else None, dres if wr else None, stats, flavour,
                     "d=%d dy2=%d dres=%d" % (d, w2, wr))


@pytest.mark.parametrize("d", [36, 1024])
@pytest.mark.parametrize("rows", [1, 7, 129, 75776, 75777])
def test_layernorm_row_partition(rows, d):
    """The backward grid is capped at 4 x 148 = 592 blocks of ceil(rows / 592) rows: 75 776 rows fill it exactly, 75 777 give 129
    rows per block and leave blocks 588-591 without rows (their partials must be exact zeros, written over a NaN workspace);
    1 and 7 rows are fewer than the row groups of one block.  dgamma / dbeta repeat bit for bit."""
    flavour = L.LN_TORCH
    x, gamma, beta, dy, dy2, dres = ln_inputs(rows, d, seed=rows + d)
    stats = ln_check_fwd("layernorm", x, gamma, beta, flavour, "rows=%d" % rows)
    (dx, dg, db), ref, bars = ln_check_bwd("layernorm", "fanout", x, gamma, beta, dy, dy2, dres, stats, flavour, "rows=%d" % rows)
    nblk, rpb, _ = ln_partition(rows, d)
    nb = lib().rbm_layernorm_ws_bytes(rows, d)
    ws = torch.full((nb // 4,), NAN, device=DEV)
    dx2, dg2, db2 = ln_bwd("fanout", x, gamma, dy, dy2, dres, stats, flavour, ws)
    assert torch.equal(dx, dx2) and torch.equal(dg, dg2) and torch.equal(db, db2), "run-to-run"
    part = ws.view(nblk, 2, d)
    empty = [b for b in range(nblk) if b * rpb >= rows]
    if rows == 75777:
        assert empty == [588, 589, 590, 591], empty
    for b in empty:
        assert bool((part[b] == 0).all()), ("partial of an empty block", b)
    G = dy.double() + dy2.double()
    contrib = torch.zeros(nblk, d, dtype=torch.float64, device=DEV).index_add_(0, torch.arange(rows, device=DEV) // rpb, G)
    _each_block_matters(contrib, bars["dbeta"], "dbeta rows=%d" % rows)


@pytest.mark.parametrize("flavour", [L.LN_TORCH, L.LN_BERT], ids=["torch", "bert"])
def test_layernorm_magnitude_1e4(flavour):
    """Rows of magnitude 1e4 (the bars scale with the data)."""
    x, gamma, beta, dy, dy2, dres = ln_inputs(500, 256, seed=11 + flavour, xscale=1e4, xshift=0.0)
    stats = ln_check_fwd("layernorm", x, gamma, beta, flavour, "1e4")
    ln_check_bwd("layernorm", "fanout", x, gamma, beta, dy, dy2, dres, stats, flavour, "1e4")


def _torch_fp32_ln(x, gamma, beta, flavour, G32, dres):
    """torch's fp32 LayerNorm on the CPU: nn.LayerNorm's kernel for TORCH; for BERT the reference module's formula in fp32 for y and
    the gradients, and nn.LayerNorm's fp32 moments (eps = 0) turned into 1 / (std_unbiased + eps) for the statistics -- torch.std
    accumulates in double on the CPU, so it is no fp32 yardstick."""
    xc, gc, bc = (t.cpu().clone().requires_grad_(True) for t in (x, gamma, beta))
    eps, d = LN_EPS[flavour], x.shape[1]
    if flavour == L.LN_TORCH:
        y, mean, rstd = torch.native_layer_norm(xc, [d], gc, bc, eps)
        mean, rstd = mean[:, 0], rstd[:, 0]
    else:
        y = oc.bert_layernorm(xc, gc, bc, eps)
        _, mean, rt = torch.native_layer_norm(xc.detach(), [d], None, None, 0.0)
        mean, rstd = mean[:, 0], 1.0 / (torch.sqrt(rt[:, 0].double() ** -2 * d / (d - 1)) + float(np.float32(eps)))
    y.backward(G32.cpu())
    return {"y": y, "mean": mean, "rstd": rstd, "dx": xc.grad + dres.cpu(), "dgamma": gc.grad, "dbeta": bc.grad}


@pytest.mark.parametrize("d", [64, 1024])
@pytest.mark.parametrize("flavour", [L.LN_TORCH, L.LN_BERT], ids=["torch", "bert"])
def test_layernorm_large_mean_small_spread(flavour, d):
    """Rows offset by 1e3 with spread 1e-2: every fp32 LayerNorm loses ~1e5 u here.  Bar per quantity: 8 x the largest error of
    torch's fp32 LayerNorm on the same input against the same float64 reference, + 2^-20 of the largest reference value."""
    x, gamma, beta, dy, dy2, dres = ln_inputs(256, d, seed=d + flavour, xscale=1e-2, xshift=1e3)
    y, stats = ln_fwd(x, gamma, beta, flavour)
    dx, dg, db = ln_bwd("fanout", x, gamma, dy, dy2, dres, stats, flavour)
    ref = ln_ref64(x, gamma, beta, flavour, dy.double() + dy2.double(), dres)
    tr = _torch_fp32_ln(x, gamma, beta, flavour, dy + dy2, dres)
    got = {"y": y, "mean": stats[:, 0], "rstd": stats[:, 1], "dx": dx, "dgamma": dg, "dbeta": db}
    for nm, v in got.items():
        rv = ref[nm]
        e_torch = float((tr[nm].detach().double().to(DEV) - rv).abs().max())
        bar = 8 * e_torch + 2.0 ** -20 * float(rv.abs().max())
        _check("layernorm_large_mean (8x torch)", v, rv, torch.full_like(rv, bar), "d=%d %s" % (d, nm))


@pytest.mark.parametrize("flavour", [L.LN_TORCH, L.LN_BERT], ids=["torch", "bert"])
def test_layernorm_autograd(flavour):
    """ops.layernorm (the autograd function the models call) against the same float64 reference."""
    x, gamma, beta, dy, _, _ = ln_inputs(129, 128, seed=5 + flavour)
    xg, gg, bg = (t.clone().requires_grad_(True) for t in (x, gamma, beta))
    y = ops.layernorm(xg, gg, bg, LN_EPS[flavour], flavour)
    y.backward(dy)
    ref = ln_ref64(x, gamma, beta, flavour, dy.double())
    bars = ln_bars(x, gamma, beta, ref, flavour, dy, depth=ln_partition(129, 128)[2])
    for nm, got in (("y", y.detach()), ("dx", xg.grad), ("dgamma", gg.grad), ("dbeta", bg.grad)):
        _check("layernorm", got, ref[nm], bars[nm], "autograd " + nm)


# ================================================================================================================ embedding
def embed_fwd(tok, table, pos, Ln, vocab, scale, zero_pad, p, shard=None):
    rows, d = tok.numel(), pos.shape[1]
    out = torch.full((rows, d), NAN, device=DEV)
    if shard is None:
        rc = lib().rbm_embed_fwd(P(tok), P(table), P(pos), P(out), rows, Ln, d, vocab, scale, zero_pad, p, SEED, SITE, S())
    else:
        v0, v1 = shard
        rc = lib().rbm_embed_fwd_shard(P(tok), P(table[v0:v1]), P(pos), P(out), rows, Ln, d, vocab, v0, v1, scale, zero_pad, p,
                                       SEED, SITE, S())
    L.check(rc, "embed_fwd")
    return out


def embed_bwd(tok, dout, Ln, zero_pad, p, row_offset=None):
    """rbm_embed_bwd, or rbm_embed_bwd_offset for a rank's slice starting at global row `row_offset`."""
    rows, d = dout.shape
    g, dpos = torch.full_like(dout, NAN), torch.full((Ln, d), NAN, device=DEV)
    if row_offset is None:
        rc = lib().rbm_embed_bwd(P(tok), P(dout), P(g), P(dpos), rows, Ln, d, zero_pad, p, SEED, SITE, S())
    else:
        rc = lib().rbm_embed_bwd_offset(P(tok), P(dout), P(g), P(dpos), rows, Ln, d, zero_pad, p, SEED, SITE, row_offset, S())
    L.check(rc, "embed_bwd")
    return g, dpos


def embed_ref64(tok, table, pos, Ln, scale, zero_pad, p):
    """(out, magnitude, bad-token rows) in float64; bad rows (token < 0 or >= vocab) must come out NaN."""
    t = tok.reshape(-1)
    rows, d = t.numel(), table.shape[1]
    bad = (t < 0) | (t >= table.shape[0])
    e = table.double()[t.clamp(0, table.shape[0] - 1)] * scale
    pe = pos.double()[torch.arange(rows, device=DEV) % Ln]
    m = _mask64(rows * d, p).view(rows, d)
    live = torch.ones(rows, 1, dtype=torch.float64, device=DEV) if not zero_pad else (t != 0).double()[:, None]
    return (e + pe) * m * live, (e.abs() + pe.abs()) * m * live, bad


def embed_grad_ref64(tok, dout, Ln, zero_pad, p):
    t = tok.reshape(-1)
    rows, d = dout.shape
    g = dout.double() * _mask64(rows * d, p).view(rows, d)
    if zero_pad:
        g = g * (t != 0).double()[:, None]
    return g, g.view(-1, Ln, d).sum(0), g.abs().view(-1, Ln, d).sum(0)


def embed_tokens(B, Ln, vocab, seed, bad=False):
    g = torch.Generator().manual_seed(seed)
    tok = torch.randint(0, vocab, (B, Ln), generator=g)
    tok[0, :Ln // 2] = 0  # a padded prefix
    tok[1, :] = 0  # an all-padding sequence
    if bad:
        tok[2, 3], tok[3, 0], tok[4, Ln - 1] = -1, vocab, vocab + 5
    return tok.to(DEV)


SHARDS = {1: [0, 50], 2: [0, 25, 50], 3: [0, 24, 25, 50], 8: [0, 7, 14, 14, 21, 28, 35, 42, 50]}  # 3: one-row shard; 8: an empty one


@pytest.mark.parametrize("p", [0.0, 0.3])
@pytest.mark.parametrize("zero_pad,scale", [(1, 6.0), (0, 1.0)])
def test_embed_fwd_shards(zero_pad, scale, p):
    """rbm_embed_fwd against float64; the sum of rbm_embed_fwd_shard over 1, 2, 3 and 8 vocabulary shards (a one-row shard and an
    empty one among them) equals it bit for bit; tokens < 0 or >= vocab give NaN rows in both."""
    B, Ln, d, vocab = 12, 20, 36, 50
    g = _gen(3)
    tok = embed_tokens(B, Ln, vocab, seed=4, bad=True)
    table, pos = torch.randn(vocab, d, device=DEV, generator=g), torch.randn(Ln, d, device=DEV, generator=g)
    full = embed_fwd(tok, table, pos, Ln, vocab, scale, zero_pad, p)
    ref, mag, bad = embed_ref64(tok, table, pos, Ln, scale, zero_pad, p)
    assert bool(full[bad].isnan().all()) and int(bad.sum()) == 3
    _check("embed", full[~bad], ref[~bad], 3 * U * mag[~bad], "fwd")
    for ns, bounds in SHARDS.items():
        total = torch.zeros_like(full)
        for v0, v1 in zip(bounds[:-1], bounds[1:]):
            total += embed_fwd(tok, table, pos, Ln, vocab, scale, zero_pad, p, shard=(v0, v1))
        assert bool(total[bad].isnan().all()), ns
        assert torch.equal(total[~bad], full[~bad]), ("shard sum", ns)


@pytest.mark.parametrize("p", [0.0, 0.3])
@pytest.mark.parametrize("zero_pad", [1, 0])
def test_embed_bwd_rank_slices(zero_pad, p):
    """rbm_embed_bwd against float64 (g, dpos); the global batch split into rank slices of 3, 1 and 36 sequences with row_offset:
    the slices' g concatenated equals the global g bit for bit (an off-by-one offset shifts the dropout stream), and the sum of the
    slices' dpos matches float64."""
    B, Ln, d = 40, 20, 36
    tok = embed_tokens(B, Ln, 50, seed=9)
    dout = torch.randn(B * Ln, d, device=DEV, generator=_gen(10))
    g, dpos = embed_bwd(tok, dout, Ln, zero_pad, p)
    g64, dpos64, dmag = embed_grad_ref64(tok, dout, Ln, zero_pad, p)
    _check("embed", g, g64, 2 * U * g64.abs(), "g")
    _check("embed", dpos, dpos64, (-(-B // 16) + 16 + 2) * U * dmag, "dpos")
    cuts = [0, 3, 4, B]
    gs, dsum = [], torch.zeros_like(dpos)
    for b0, b1 in zip(cuts[:-1], cuts[1:]):
        gi, di = embed_bwd(tok[b0:b1].contiguous(), dout[b0 * Ln:b1 * Ln].contiguous(), Ln, zero_pad, p, row_offset=b0 * Ln)
        gs.append(gi)
        dsum += di
    assert torch.equal(torch.cat(gs), g), "slices of the global g"
    _check("embed", dsum, dpos64, (-(-B // 16) + 16 + len(cuts) + 2) * U * dmag, "sliced dpos")


@pytest.mark.parametrize("p", [0.0, 0.25])
@pytest.mark.parametrize("zero_pad,scale", [(1, 8.0), (0, 1.0)])
def test_embed_autograd(zero_pad, scale, p):
    """ops.EmbedFn forward and backward (table gradient through the sorted scatter, positional gradient) against float64."""
    B, Ln, d, vocab = 5, 12, 32, 41
    g = _gen(21)
    tok = embed_tokens(B, Ln, vocab, seed=22)
    table, pos = torch.randn(vocab, d, device=DEV, generator=g), torch.randn(Ln, d, device=DEV, generator=g)
    dout = torch.randn(B * Ln, d, device=DEV, generator=g)
    tg, pg = table.clone().requires_grad_(True), pos.clone().requires_grad_(True)
    out = ops.EmbedFn.apply(tok, tg, pg, scale, zero_pad, p, SEED, SITE)
    out.backward(dout.view(B, Ln, d))
    ref, mag, _ = embed_ref64(tok, table, pos, Ln, scale, zero_pad, p)
    _check("embed", out.detach().view(-1, d), ref, 3 * U * mag, "autograd out")
    g64, dpos64, dmag = embed_grad_ref64(tok, dout, Ln, zero_pad, p)
    _check("embed", pg.grad, dpos64, (-(-B // 16) + 16 + 2) * U * dmag, "autograd dpos")
    t = tok.reshape(-1)
    keep = t != 0  # the table's padding row receives nothing (padding_idx = 0)
    dt64 = torch.zeros(vocab, d, dtype=torch.float64, device=DEV).index_add_(0, t[keep], scale * g64[keep])
    dtm = torch.zeros(vocab, d, dtype=torch.float64, device=DEV).index_add_(0, t[keep], scale * g64[keep].abs())
    cnt = torch.bincount(t[keep], minlength=vocab).double()[:, None]
    _check("embed", tg.grad, dt64, (cnt + 3) * U * dtm, "autograd dtable")


def embed_bwd_rows(tok, rows, count, cap, dout_c, Ln, p):
    d = dout_c.shape[1]
    g_c = torch.full((cap, d), NAN, device=DEV)
    idx_c = torch.full((cap,), -7, dtype=torch.int64, device=DEV)
    dpos = torch.full((Ln, d), NAN, device=DEV)
    nb = lib().rbm_embed_bwd_rows_ws_bytes(Ln, d)
    ws = torch.full((nb // 4,), NAN, device=DEV)
    rc = lib().rbm_embed_bwd_rows(P(tok), P(rows), P(count), cap, P(dout_c), P(g_c), P(idx_c), P(dpos), Ln, d, p, SEED, SITE, P(ws), nb,
                                  S())
    return rc, g_c, idx_c, dpos


def live_rows(tok, cap):
    """rows [max(n, cap)] int32 (ascending live row ids, zeros after them) and count, built on the host side from the tokens."""
    flat = tok.reshape(-1)
    live = (flat != 0).nonzero()[:, 0].to(torch.int32)
    n = int(live.numel())
    rows = torch.zeros(max(flat.numel(), cap), dtype=torch.int32, device=DEV)
    rows[:n] = live
    return rows, torch.tensor([n], dtype=torch.int32, device=DEV), n


def check_embed_bwd_rows(tok, Ln, d, cap_extra, p, seed):
    rows, count, n = live_rows(tok, 0)
    cap = max(n + cap_extra, 1)
    if cap > rows.numel():
        rows = torch.cat([rows, torch.zeros(cap - rows.numel(), dtype=torch.int32, device=DEV)])
    dout_c = torch.rand(cap, d, device=DEV, generator=_gen(seed)) + 0.25  # positive: every dpos partial block shows (see below)
    rc, g_c, idx_c, dpos = embed_bwd_rows(tok, rows, count, cap, dout_c, Ln, p)
    L.check(rc, "embed_bwd_rows")
    r = rows[:n].long()
    # g_c is the gather of rbm_embed_bwd's g (zero_pad = 1) for the same upstream gradient
    dout_full = torch.zeros(tok.numel(), d, device=DEV)
    dout_full[r] = dout_c[:n]
    g_full, _ = embed_bwd(tok, dout_full, Ln, 1, p)
    assert torch.equal(g_c[:n], g_full[r]), "g_c vs rbm_embed_bwd"
    assert bool((g_c[n:] == 0).all()) and bool((idx_c[n:] == 0).all()), "rows past count"
    assert torch.equal(idx_c[:n], tok.reshape(-1)[r])
    g64 = dout_c[:n].double() * _mask64(tok.numel() * d, p).view(-1, d)[r]
    _check("embed_rows", g_c[:n], g64, 2 * U * g64.abs(), "g_c")
    l = r % Ln
    dpos64 = torch.zeros(Ln, d, dtype=torch.float64, device=DEV).index_add_(0, l, g64)
    per = -(-n // NSM)
    bar = (per + NSM + 2) * U * torch.zeros_like(dpos64).index_add_(0, l, g64.abs())
    _check("embed_rows", dpos, dpos64, bar, "dpos L=%d d=%d" % (Ln, d))
    if n:
        blk = torch.arange(n, device=DEV) // per
        contrib = torch.zeros(NSM, Ln, d, dtype=torch.float64, device=DEV).index_put_((blk, l), g64, accumulate=True)
        _each_block_matters(contrib, bar, "dpos")


# (L, d): d / 4 = 16, 64, 256 -> 32, 64, 128 threads per dpos block; no shape here needs opt-in shared memory
@pytest.mark.parametrize("Ln,d", [(50, 64), (40, 256), (20, 1024)])
@pytest.mark.parametrize("kind", ["spare_cap", "full_cap", "all_padding"])
def test_embed_bwd_rows(kind, Ln, d):
    """rbm_embed_bwd_rows: g_c, idx_c and dpos against float64 and g_c against rbm_embed_bwd's g bit for bit, with cap > count (the
    rows past count must be zeros, idx_c 0 there), cap = count, and count = 0."""
    B = 64
    tok = embed_tokens(B, Ln, 300, seed=Ln + d)
    if kind == "all_padding":
        tok.zero_()
    check_embed_bwd_rows(tok, Ln, d, {"spare_cap": 37, "full_cap": 0, "all_padding": 16}[kind], 0.3, seed=d)


def test_embed_bwd_rows_image_sizes():
    """The [L, d] positional image in shared memory: 200 x 64 floats = 51 200 B needs the opt-in limit, then 192 x 128 = 96 KB
    exactly (a larger image after a smaller one: the cached limit must be raised again); 193 x 128 is refused before any launch."""
    for Ln, d in ((200, 64), (192, 128)):
        check_embed_bwd_rows(embed_tokens(24, Ln, 300, seed=Ln), Ln, d, 5, 0.0, seed=Ln)
    tok = embed_tokens(4, 193, 300, seed=1)
    rows, count, n = live_rows(tok, 0)
    rc, *_ = embed_bwd_rows(tok, rows, count, n, torch.zeros(n, 128, device=DEV), 193, 0.0)
    assert rc < 0 and b"96 KB" in lib().rbm_last_error()


# ============================================================================================================= row layouts
def seq_start(rows, count, B, Ln):
    ss = torch.full((B + 1,), -5, dtype=torch.int32, device=DEV)
    L.check(lib().rbm_rows_seq_start(P(rows), P(count), B, Ln, P(ss), S()), "rows_seq_start")
    return ss


@pytest.mark.parametrize("case", ["mixed_spare_cap", "mixed_full_cap", "all_padding"])
def test_rows_layouts(case):
    """rbm_rows_seq_start, rbm_rows_to_seq and rbm_seq_to_rows against a reference built from the token matrix (sequences without
    live rows, sequences with exactly Lq live rows, an all-padding batch, cap > count), bit for bit, and their adjointness in
    float64; rbm_rows_gather with a coefficient that zeroes a row."""
    B, Ln, Lq, d = 9, 12, 5, 36
    counts = [0, 5, 3, 0, 1, 5, 2, 4, 0] if case != "all_padding" else [0] * B
    g = torch.Generator().manual_seed(len(case))
    tok = torch.zeros(B, Ln, dtype=torch.long)
    for b, c in enumerate(counts):
        tok[b, torch.randperm(Ln, generator=g)[:c]] = torch.randint(1, 100, (c,), generator=g)
    tok = tok.to(DEV)
    n = sum(counts)
    cap = n + 7 if case != "mixed_full_cap" else n
    cap = max(cap, 1)
    rows, count, _ = live_rows(tok, cap)
    ss = seq_start(rows, count, B, Ln)
    ref_ss = torch.tensor(np.concatenate([[0], np.cumsum(counts)]), dtype=torch.int32, device=DEV)
    assert torch.equal(ss, ref_ss), (ss, ref_ss)

    x = torch.randn(cap, d, device=DEV, generator=_gen(1))
    to_seq = torch.full((B * Lq, d), NAN, device=DEV)
    L.check(lib().rbm_rows_to_seq(P(x), P(ss), B, Lq, d, P(to_seq), S()), "rows_to_seq")
    ref = torch.zeros(B * Lq, d, device=DEV)
    for b in range(B):
        c = counts[b]
        ref[b * Lq:b * Lq + c] = x[int(ref_ss[b]):int(ref_ss[b]) + c]
    assert torch.equal(to_seq, ref), "rows_to_seq"

    y = torch.randn(B * Lq, d, device=DEV, generator=_gen(2))
    back = torch.full((cap, d), NAN, device=DEV)
    L.check(lib().rbm_seq_to_rows(P(y), P(rows), P(ss), P(count), cap, Ln, Lq, d, P(back), S()), "seq_to_rows")
    ref = torch.zeros(cap, d, device=DEV)
    for b in range(B):
        c = counts[b]
        ref[int(ref_ss[b]):int(ref_ss[b]) + c] = y[b * Lq:b * Lq + c]
    assert torch.equal(back, ref), "seq_to_rows"
    lhs = float((to_seq.double() * y.double()).sum())
    rhs = float((x.double() * back.double()).sum())
    assert abs(lhs - rhs) <= 2.0 ** -40 * float((to_seq.double() * y.double()).abs().sum()), (lhs, rhs)

    src = torch.randn(B * Ln, d + 8, device=DEV, generator=_gen(3))  # row stride d + 8
    coef = torch.randn(B * Ln, device=DEV, generator=_gen(4))
    if n:
        coef[rows[1].long()] = 0.0
    dst = torch.full((cap, d), NAN, device=DEV)
    L.check(lib().rbm_rows_gather(P(src), d + 8, P(rows), P(count), cap, d, P(coef), P(dst), S()), "rows_gather")
    ref = torch.zeros(cap, d, device=DEV)
    r = rows[:n].long()
    ref[:n] = coef[r][:, None] * src[r, :d]
    assert torch.equal(dst, ref), "rows_gather"


def colsum_call(which, src, ld, key, n, d):
    """rbm_rows_dead_colsum (key = tok, n rows) or rbm_rows_live_colsum (key = count, cap = n) on a NaN workspace and output."""
    nb = lib().rbm_rows_dead_colsum_ws_bytes(d)
    ws = torch.full((nb // 4,), NAN, device=DEV)
    out = torch.full((d,), NAN, device=DEV)
    fn = lib().rbm_rows_dead_colsum if which == "dead" else lib().rbm_rows_live_colsum
    L.check(fn(P(src), ld, P(key), n, d, P(out), P(ws), nb, S()), which + "_colsum")
    return out


# n = 47 357: ceil(n / 1184) = 40 rows per block and the last block starts at 47 320 < n -- every one of the 1184 blocks has rows
@pytest.mark.parametrize("n,d", [(0, 64), (1000, 48), (1000, 1024), (47357, 64)])
@pytest.mark.parametrize("which", ["dead", "live"])
def test_rows_colsums(which, n, d):
    """rbm_rows_dead_colsum (rows with tok == 0) and rbm_rows_live_colsum (the first count rows) against float64: n = 0, d = 48
    (4 threads of each block idle), d = 1024 (one row lane), and n large enough that all 1184 partial blocks have rows.  Repeats
    bit for bit."""
    ld = d + 8
    g = _gen(n + d)
    src = torch.rand(max(n, 1) + 3, ld, device=DEV, generator=g) + 0.5  # positive: every partial block's share shows
    if which == "dead":
        key = (torch.rand(max(n, 1), device=DEV, generator=g) < 0.4).long() * 7  # 60 % padding rows
        sel = key[:n] == 0
        cnt = n
    else:
        cnt = max(n - 13, 0)
        key = torch.tensor([cnt], dtype=torch.int32, device=DEV)
        sel = torch.arange(n, device=DEV) < cnt
    out = colsum_call(which, src, ld, key, n, d)
    out2 = colsum_call(which, src, ld, key, n, d)
    assert torch.equal(out, out2), "run-to-run"
    terms = src[:n, :d].double() * sel.double()[:, None]
    ref = terms.sum(0)
    nro = 256 // (d // 4)
    per = -(-n // 1184)
    bar = (-(-per // nro) + nro + 5 + 8 + 2) * U * terms.abs().sum(0)
    _check("rows_colsum", out, ref, bar, "%s n=%d d=%d" % (which, n, d))
    if n:
        contrib = torch.zeros(1184, d, dtype=torch.float64, device=DEV).index_add_(0, torch.arange(n, device=DEV) // per, terms)
        _each_block_matters(contrib, bar, "%s colsum" % which)
        if n == 47357:
            assert bool((contrib.abs().sum(1) > 0).all()), "every block has rows"


# ======================================================================================================= SASRec scoring, BCE
def pick_gw(d):
    d4 = d // 4
    return 4 if d4 <= 4 else 8 if d4 <= 8 else 16 if d4 <= 16 else 32


def dot_bar(d, mag):
    gw = pick_gw(d)
    return (-(-(d // 4) // gw) + int(math.log2(gw)) + 4) * U * mag


def sas_inputs(rows, d, V, seed):
    g = _gen(seed)
    f = torch.randn(rows, d, device=DEV, generator=g)
    table = torch.randn(V, d, device=DEV, generator=g) * 0.3
    pos = torch.randint(1, V, (rows,), device=DEV, generator=g)
    pos[::3] = 0
    neg = torch.randint(1, V, (rows,), device=DEV, generator=g)
    return f, table, pos, neg


# d = 16 / 20 / 32 / 36 / 64 / 68 / 128 / 256 / 1024 -> gw = 4, 8, 8, 16, 16, 32, 32, 32, 32; 1001 rows: not a multiple of 256 / gw
@pytest.mark.parametrize("d", [16, 20, 32, 36, 64, 68, 128, 256, 1024])
def test_sas_score(d):
    """rbm_sas_score_fwd (pl, nl) and rbm_sas_score_bwd (df) against float64."""
    rows, V = 1001, 3000
    f, table, pos, neg = sas_inputs(rows, d, V, seed=d)
    pl, nl = torch.full((rows,), NAN, device=DEV), torch.full((rows,), NAN, device=DEV)
    L.check(lib().rbm_sas_score_fwd(P(f), P(table), P(pos), P(neg), P(pl), P(nl), rows, d, S()), "sas_score_fwd")
    f64, tp, tn = f.double(), table.double()[pos], table.double()[neg]
    _check("sas_score", pl, (f64 * tp).sum(1), dot_bar(d, (f64 * tp).abs().sum(1)), "pl d=%d" % d)
    _check("sas_score", nl, (f64 * tn).sum(1), dot_bar(d, (f64 * tn).abs().sum(1)), "nl d=%d" % d)
    g = _gen(d + 1)
    dpl, dnl = torch.randn(rows, device=DEV, generator=g), torch.randn(rows, device=DEV, generator=g)
    df = torch.full_like(f, NAN)
    L.check(lib().rbm_sas_score_bwd(P(table), P(pos), P(neg), P(dpl), P(dnl), P(df), rows, d, S()), "sas_score_bwd")
    a, b = dpl.double()[:, None] * tp, dnl.double()[:, None] * tn
    _check("sas_score", df, a + b, 2 * U * (a.abs() + b.abs()), "df d=%d" % d)


@pytest.mark.parametrize("ids", ["disjoint", "shared"])
def test_sas_score_table_gradient(ids):
    """The table gradient of ops.sas_scores with cap=None (two scatters) and with cap (one sort over the compacted positive and
    negative entries) against float64, and f's gradient against rbm_sas_score_bwd.  With disjoint positive and negative ids every
    table row gets its contributions in the same order on both paths, so they agree bit for bit; when an id is in both lists the
    cap path adds them in one chain, (P + n1) + n2 instead of P + (n1 + n2), so there both are held to the float64 bar only.
    Id 5 is hot (more than 64 contributions: the multi-piece scatter)."""
    rows, d, V = 3000, 64, 2000
    f, table, pos, neg = sas_inputs(rows, d, V, seed=len(ids))
    if ids == "disjoint":
        pos = torch.where(pos == 0, pos, pos % 999 + 1)  # 1..999
        neg = neg % 1000 + 1000  # 1000..1999
        pos[1::7] = 5
    else:
        pos[1::7] = 5
        neg[::11] = 5
    g = _gen(7)
    wp, wn = torch.randn(rows, device=DEV, generator=g), torch.randn(rows, device=DEV, generator=g)
    cap = max(int((pos != 0).sum()), int((neg != 0).sum())) + 3
    grads = []
    for c in (None, cap):
        fg, tg = f.clone().requires_grad_(True), table.clone().requires_grad_(True)
        pl, nl = ops.sas_scores(fg, tg, pos, neg, cap=c)
        (pl * wp + nl * wn).sum().backward()
        grads.append((fg.grad, tg.grad))
    df = torch.empty_like(f)
    L.check(lib().rbm_sas_score_bwd(P(table), P(pos), P(neg), P(wp), P(wn), P(df), rows, d, S()), "sas_score_bwd")
    assert torch.equal(grads[0][0], df) and torch.equal(grads[1][0], df)
    f64 = f.double()
    ref = torch.zeros(V, d, dtype=torch.float64, device=DEV)
    mag = torch.zeros_like(ref)
    cnt = torch.zeros(V, dtype=torch.float64, device=DEV)
    for idx, w in ((pos, wp), (neg, wn)):
        k = idx != 0
        t = w.double()[k, None] * f64[k]
        ref.index_add_(0, idx[k], t)
        mag.index_add_(0, idx[k], t.abs())
        cnt.index_add_(0, idx[k], torch.ones_like(t[:, 0]))
    bar = (cnt[:, None] + 3) * U * mag
    for c, (_, dt) in zip(("cap=None", "cap"), grads):
        _check("sas_score", dt, ref, bar, "dtable " + c)
    if ids == "disjoint":
        assert torch.equal(grads[0][1], grads[1][1]), "cap path vs cap=None"


def bce_call(pl, nl, pos, dloss=1.0):
    rows = pl.numel()
    nb = lib().rbm_bce_ws_bytes(rows)
    ws = torch.full((nb // 4,), NAN, device=DEV)
    loss = torch.full((1,), NAN, device=DEV)
    count = torch.full((1,), -3, dtype=torch.int32, device=DEV)
    L.check(lib().rbm_bce_pair_fwd(P(pl), P(nl), P(pos), P(loss), P(count), rows, P(ws), nb, S()), "bce_fwd")
    dl = torch.full((1,), dloss, device=DEV)
    dpl, dnl = torch.full_like(pl, NAN), torch.full_like(nl, NAN)
    L.check(lib().rbm_bce_pair_bwd(P(pl), P(nl), P(pos), P(count), P(dl), P(dpl), P(dnl), rows, S()), "bce_bwd")
    return loss, count, dpl, dnl


def _softplus64(z):
    return z.clamp(min=0) + torch.log1p(torch.exp(-z.abs()))


@pytest.mark.parametrize("rows", [1023, 1024, 1025, 204800])
def test_bce(rows):
    """rbm_bce_pair_fwd / _bwd against float64 around the 1024-row partial blocks, with logits of +-100 (softplus and sigmoid
    saturate); the loss repeats bit for bit."""
    g = _gen(rows)
    pl = torch.randn(rows, device=DEV, generator=g) * 3
    nl = torch.randn(rows, device=DEV, generator=g) * 3
    pl[::97], nl[5::89], pl[7::101], nl[3::103] = 100.0, 100.0, -100.0, -100.0
    pos = torch.randint(1, 50, (rows,), device=DEV, generator=g)
    pos[torch.rand(rows, device=DEV, generator=g) < 0.25] = 0
    loss, count, dpl, dnl = bce_call(pl, nl, pos)
    loss2, *_ = bce_call(pl, nl, pos)
    assert torch.equal(loss, loss2), "run-to-run"
    on = (pos != 0).double()
    c = int(on.sum())
    assert int(count) == c
    sp, sn = _softplus64(-pl.double()) * on, _softplus64(nl.double()) * on
    terms = sp + sn
    ref = float(terms.sum()) / c
    nblk = -(-rows // 1024)
    bar = (4 + 8 + nblk + 8) * U * float(terms.sum()) / c
    _check("bce", loss, torch.tensor([ref], dtype=torch.float64, device=DEV), torch.tensor([bar], device=DEV, dtype=torch.float64),
           "loss rows=%d" % rows)
    contrib = torch.zeros(nblk, dtype=torch.float64, device=DEV).index_add_(0, torch.arange(rows, device=DEV) // 1024, terms) / c
    _each_block_matters(contrib[:, None], torch.tensor([bar], dtype=torch.float64, device=DEV), "bce loss")
    gs = 1.0 / c
    sp_, sn_ = torch.sigmoid(pl.double()), torch.sigmoid(nl.double())
    _check("bce", dpl, gs * (sp_ - 1) * on, (8 * U * gs * (sp_ + (1 - sp_).abs()) + 2.0 ** -126 * gs) * on, "dpl")
    _check("bce", dnl, gs * sn_ * on, (8 * U * gs * sn_ + 2.0 ** -126 * gs) * on, "dnl")
    assert bool((dpl[pos == 0] == 0).all()) and bool((dnl[pos == 0] == 0).all())


def test_bce_no_positive_row():
    """No row with pos != 0: count is 0, the loss is NaN (the reference's mean over no rows) and both gradients are exact zeros."""
    rows = 3000
    g = _gen(1)
    loss, count, dpl, dnl = bce_call(torch.randn(rows, device=DEV, generator=g), torch.randn(rows, device=DEV, generator=g),
                                     torch.zeros(rows, dtype=torch.int64, device=DEV))
    assert int(count) == 0 and bool(torch.isnan(loss).all())
    assert bool((dpl == 0).all()) and bool((dnl == 0).all())


# (U, C, d, bias): d = 64 -> 16 rows per block, 37 * 101 = 3737 is not a multiple; C = 1; d = 1024 -> 8 per block, 13 * 7 = 91
@pytest.mark.parametrize("U_,C,d,bias", [(37, 101, 64, True), (37, 101, 64, False), (1000, 1, 36, True), (13, 7, 1024, False)])
def test_candidate_scores(U_, C, d, bias):
    """ops.candidate_scores / rbm_candidate_scores on a strided f (row stride d + 12) against float64, with and without bias."""
    V = 500
    g = _gen(U_ + C + d)
    base = torch.randn(U_, d + 12, device=DEV, generator=g)
    f = base[:, :d]
    table = torch.randn(V, d, device=DEV, generator=g)
    b = torch.randn(V, device=DEV, generator=g) if bias else None
    cand = torch.randint(0, V, (U_, C), device=DEV, generator=g)
    out = torch.full((U_, C), NAN, device=DEV)
    L.check(lib().rbm_candidate_scores(P(f), d + 12, P(table), P(b), P(cand), P(out), U_, C, d, S()), "candidate_scores")
    assert torch.equal(ops.candidate_scores(f, table, b, cand), out)  # the wrapper passes the view's row stride through
    prod = table.double()[cand] * f.double()[:, None, :]
    ref = prod.sum(-1) + (b.double()[cand] if bias else 0.0)
    mag = prod.abs().sum(-1) + (b.double()[cand].abs() if bias else 0.0)
    _check("candidate_scores", out, ref, dot_bar(d, mag), "U=%d C=%d d=%d" % (U_, C, d))


# ================================================================================================= metric means, Adam, bucket
def column_mean(x):
    Un, cols = x.shape
    nb = lib().rbm_column_mean_ws_bytes(Un, cols)
    ws = torch.full((nb // 4,), NAN, device=DEV)
    out = torch.full((cols,), NAN, device=DEV)
    L.check(lib().rbm_column_mean(P(x), P(out), Un, cols, P(ws), nb, S()), "column_mean")
    return out


# 4096 rows per block; 4 194 305 rows pass 1024 blocks (the grid is capped there, 4097 rows per block)
@pytest.mark.parametrize("cols", [1, 256])
@pytest.mark.parametrize("Un", [1, 4096, 4097, 4194305])
def test_column_mean(Un, cols):
    """rbm_column_mean within 1 fp32 ulp of the exact mean; repeats bit for bit."""
    x = torch.rand(Un, cols, device=DEV, generator=_gen(Un + cols))
    out = column_mean(x)
    assert torch.equal(out, column_mean(x)), "run-to-run"
    s = x.double().sum(0)
    ref = s / Un
    r32 = ref.float()
    ulp = (torch.nextafter(r32, torch.full_like(r32, math.inf)) - r32).double()
    _check("column_mean (1 ulp)", out, ref, ulp, "U=%d cols=%d" % (Un, cols))
    nblk = min(max(-(-Un // 4096), 1), 1024)
    rpb = -(-Un // nblk)
    contrib = torch.zeros(nblk, cols, dtype=torch.float64, device=DEV).index_add_(0, torch.arange(Un, device=DEV) // rpb, x.double())
    _each_block_matters(contrib / Un, ulp, "column mean")


ADAM_SIZES = [1, 3, 4, 4095, 4096, 4097]


def adam_tensors(sizes, seed, misaligned_last=False):
    """Per tensor (p, g, m, v) fp32 CUDA tensors; with misaligned_last one more tensor of 4097 elements whose four pointers all sit
    4 bytes past a 16-byte boundary (the kernel's scalar path)."""
    g = _gen(seed)
    out = []
    for n in sizes:
        out.append([torch.randn(n, device=DEV, generator=g), None, torch.randn(n, device=DEV, generator=g) * 0.1,
                    torch.rand(n, device=DEV, generator=g) * 0.01])
    if misaligned_last:
        views = []
        for k in range(4):
            st = torch.empty(4098, device=DEV)
            v = st[1:]
            v.copy_(torch.randn(4097, device=DEV, generator=g) if k != 3 else torch.rand(4097, device=DEV, generator=g) * 0.01)
            assert v.data_ptr() % 16 == 4
            views.append(v)
        out.append(views)
    return out


def adam_call(ts, step, lr, wd, b1=0.9, b2=0.999, eps=1e-8):
    desc = torch.tensor([[p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel()] for p, g, m, v in ts], dtype=torch.int64)
    desc = desc.to(DEV)
    cmap = rd.chunk_map([p.numel() for p, *_ in ts]).to(DEV)
    L.check(lib().rbm_adam_multi(P(desc), P(cmap), cmap.shape[0], lr, b1, b2, eps, wd, step, S()), "adam_multi")
    torch.cuda.synchronize()


def _adam_bound(p, g, m, v, E, step, lr, wd, b1=0.9, b2=0.999, eps=1e-8):
    """One step of the float64 reference (oracle.optim.adam_step on float64 arrays, same fp32 constants) together with a first-order
    bound E = (Ep, Em, Ev) on the fp32 kernel's distance from it: one rounding u per operation on the operation's magnitude."""
    f = np.float32
    Ep, Em, Ev = E
    c1, c2 = float(f(1.0 - b1)), float(f(1.0 - b2))
    gg = g + float(f(wd)) * p
    Eg = float(f(wd)) * Ep + U * (np.abs(g) + float(f(wd)) * np.abs(p))
    Em = (1 - c1) * Em + c1 * Eg + 2 * U * (np.abs(m) + np.abs(gg))
    Ev = float(f(b2)) * Ev + 2 * c2 * np.abs(gg) * Eg + 3 * U * (float(f(b2)) * v + c2 * gg * gg)
    oo.adam_step(p, g, m, v, step, lr, b1, b2, eps, wd)  # p, m, v now the float64 state after this step
    ss = float(f(lr / (1.0 - b1 ** step)))
    den = np.sqrt(v) / float(f(math.sqrt(1.0 - b2 ** step))) + float(f(eps))
    rho = np.where(v > 0, Ev / np.where(v > 0, v, 1.0), 0.0) / 2 + 4 * U  # relative error of the denominator
    upd = np.abs(m) / den
    Ep = Ep + ss * (Em / den + upd * (rho + U)) + U * (np.abs(p) + ss * upd)
    return Ep, Em, Ev


@pytest.mark.parametrize("wd", [0.0, 0.01])
def test_adam_multi(wd):
    """rbm_adam_multi through the C ABI, four steps, against the float64 reference within the propagated bound (x2): n = 1, 3, 4,
    4095, 4096, 4097 (vector path, ragged tails, chunk edges) and one tensor with every pointer 4 bytes off (scalar path)."""
    ts = adam_tensors(ADAM_SIZES, seed=int(wd * 1000) + 1, misaligned_last=True)
    ref = [[t.double().cpu().numpy() for t in (p, m, v)] for p, _, m, v in ts]
    E = [(np.zeros(p.numel()),) * 3 for p, *_ in ts]
    lr = 1e-3
    g = _gen(99)
    for step in range(1, 5):
        for k, t in enumerate(ts):
            gr = torch.randn(t[0].numel(), device=DEV, generator=g)
            if t[0].data_ptr() % 16 == 4:
                st = torch.empty(gr.numel() + 1, device=DEV)
                st[1:].copy_(gr)
                gr = st[1:]
            t[1] = gr
            pr, mr, vr = ref[k]
            E[k] = _adam_bound(pr, gr.double().cpu().numpy(), mr, vr, E[k], step, lr, wd)
        adam_call(ts, step, lr, wd)
    for k, (p, _, m, v) in enumerate(ts):
        pr, mr, vr = (torch.from_numpy(a).to(DEV) for a in ref[k])
        Ep, Em, Ev = (torch.from_numpy(np.asarray(a)).to(DEV) for a in E[k])
        what = "n=%d%s" % (p.numel(), " misaligned" if p.data_ptr() % 16 else "")
        _check("adam", p, pr, 2 * Ep, what + " p")
        _check("adam", m, mr, 2 * Em, what + " m")
        _check("adam", v, vr, 2 * Ev, what + " v")


@pytest.mark.parametrize("s", [2, 7, 1000])
def test_adam_device_step_counter(s):
    """rbm_set_step_counter pointing at a device value of s - 1 with step = 1 equals the eager step s bit for bit (include/rbm.h)."""
    a = adam_tensors([4097, 5], seed=s)
    for ts in a:
        ts[1] = torch.randn(ts[0].numel(), device=DEV, generator=_gen(s + ts[0].numel()))
    b = [[t.clone() for t in ts] for ts in a]
    adam_call(a, s, 1e-3, 0.01)
    counter = torch.tensor([s - 1], dtype=torch.int64, device=DEV)
    try:
        L.check(lib().rbm_set_step_counter(P(counter)), "set_step_counter")
        adam_call(b, 1, 1e-3, 0.01)
    finally:
        L.check(lib().rbm_set_step_counter(None), "set_step_counter(NULL)")
    for ta, tb in zip(a, b):
        for k in (0, 2, 3):
            assert torch.equal(ta[k], tb[k]), (s, k)


def test_bucket_pack_round_trip():
    """rbm_bucket_pack / unpack at ragged (unaligned) offsets: packing with scale 1/2 stores t / 2 exactly and leaves the gaps alone,
    unpacking with scale 2 restores t bit for bit; the same with scale 1 both ways."""
    sizes = [1, 3, 4097, 5000, 8193]
    offsets = [0, 2, 9, 4110, 9115]
    total = offsets[-1] + sizes[-1] + 3
    g = _gen(5)
    ts = [torch.randn(n, device=DEV, generator=g) for n in sizes]
    orig = [t.clone() for t in ts]
    desc = torch.tensor([[t.data_ptr(), n, o] for t, n, o in zip(ts, sizes, offsets)], dtype=torch.int64).to(DEV)
    cmap = rd.chunk_map(sizes).to(DEV)
    inside = torch.zeros(total, dtype=torch.bool, device=DEV)
    for n, o in zip(sizes, offsets):
        inside[o:o + n] = True
    for scale in (0.5, 1.0):
        bucket = torch.full((total,), 1234.5, device=DEV)
        L.check(lib().rbm_bucket_pack(P(desc), P(cmap), cmap.shape[0], P(bucket), scale, 0, S()), "bucket_pack")
        for t, n, o in zip(orig, sizes, offsets):
            assert torch.equal(bucket[o:o + n], t * scale), (scale, n)
        assert bool((bucket[~inside] == 1234.5).all()), "gaps"
        for t in ts:
            t.fill_(NAN)
        L.check(lib().rbm_bucket_pack(P(desc), P(cmap), cmap.shape[0], P(bucket), 1.0 / scale, 1, S()), "bucket_unpack")
        for t, o in zip(ts, orig):
            assert torch.equal(t, o), scale
