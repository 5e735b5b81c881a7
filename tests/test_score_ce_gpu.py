"""Fused scoring + masked cross-entropy (rbm_compact_labels, rbm_ce_fwd / rbm_ce_bwd) against the float64 oracle
(oracle/common.masked_ce64), called through the C ABI so that the per-row log-sum-exp of every compacted row is checked next to
the loss, dH, dW and db.  Three kernel families sit behind one entry point (csrc/score_ce.cu):

  * tcgen05 3xTF32 (ce_tc.cu)       d in {32, 64},   V1 >= 64
  * split-fp16 tcgen05 (ce_wide.cu) d in {128, 256}, V1 >= 64
  * SIMT mma.sync (score_ce.cu)     everything else, ce_bwd_*_kernel<DT> with DT = 4 / 8 / 16 / 32 by d

Covered here: which family each shape reaches, tile and split edges of every family (row counts around 128, vocabularies around
the 64- and 128-row tiles, the device-side vocabulary split of ce_wide.cu), vocabulary shards with targets outside the shard and
the global log-sum-exp in the backward, null and unaligned bias, a bias spread of +-60, stale workspace and outputs, run-to-run
determinism and batches without a labelled row.  Run with -m gpu on a B200; `pytest -s` prints the largest error per path.

Bars (every comparison against float64), with A_r = max_v sum_k |h_rk w_vk| the logit scale of row r:
  * per-row LSE: |lse - ref| <= 2^-20 * A_r + 2^-21 * max(1, |ref|).  A product of 3xTF32 / three-pass split fp16 is good to
    2^-21 |h_k w_k|; the tensor cores then accumulate the logit in fp32 over d/8 (TF32) or d/16 (fp16) steps per pass, each step
    aligning its products to the largest exponent and truncating, so the sum also drifts by up to 2^-24 of the running |logit| per
    step, one-signed.  At d = 256 (48 fp16 steps) with logits of 20 (A_r ~ 60) that drift is 2^-19.5 of the logit, measured on a
    B200 as 1.04 x 2^-21 A_r (tests/test_kernels_gpu.py::test_score_ce): hence 2^-20 A_r.  The log-sum-exp itself is an fp32
    result of ex2 / lg2 sums: 2^-21 of its magnitude.
  * loss: 1e-6 * max(1, |ref|) + 2^-21 * mean_r A_r: the mean of lse - target logit, whose target logit carries the same
    accumulation drift (averaged over the rows).
  * dH: max |error| <= 5e-5 * max |ref|; dW, db: 2e-5 * max |ref| (tightened from 1e-4: the largest measured on a B200 are
    2.1e-5 for dH on the tcgen05 path and 8.5e-6 for dW on the split-fp16 path).
"""
import math
import re
from collections import defaultdict

import pytest
import torch

from rbm_b200 import dist as rd, ops, lib as L
from oracle import common as oc

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0)

SIMT = ("ce_fwd_kernel", "ce_bwd_dh_kernel", "ce_bwd_dw_kernel")
TC = ("ce_fwd_tc_kernel", "ce_bwd_dh_tc_kernel", "ce_bwd_dw_tc_kernel")
WIDE = ("ce_wide_fwd128_kernel", "ce_wide_kernel", "fwd_combine_kernel", "dh_reduce_kernel")
FAMILY = {"simt": SIMT, "tc": TC, "wide": WIDE}

LOSS_BAR, GRAD_BAR = 1e-6, {"dH": 5e-5, "dW": 2e-5, "db": 2e-5}
WORST = defaultdict(lambda: defaultdict(float))  # path -> quantity -> largest error / its bar scale


def path_of(V1, d):
    """The family csrc/score_ce.cu picks for aligned operands (test_ce_dispatch_reaches_every_path pins this)."""
    if V1 >= 64 and d in (32, 64):
        return "tc"
    if V1 >= 64 and d in (128, 256):
        return "wide"
    return "simt"


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    print("\nlargest error per path (lse, loss: / their bound; gradients: / max |ref|)")
    for p in sorted(WORST):
        print("  %-5s " % p + "  ".join("%s %.3g" % kv for kv in sorted(WORST[p].items())))


# ------------------------------------------------------------------------------------------------ C ABI calls
class Run:
    """What one masked cross-entropy call returns: lse [count] of the compacted rows, loss, dH, dW, db."""

    def __init__(self, lse, loss, dh, dw, db):
        self.lse, self.loss, self.dh, self.dw, self.db = lse, loss, dh, dw, db

    def tensors(self):
        return self.lse, self.loss, self.dh, self.dw, self.db


def _stale(ws):
    ws.fill_(0xFF)  # every float of it a NaN


def compact(labels, stale=False):
    lib = L.load()
    n = labels.numel()
    rows = torch.empty(n, device=DEV, dtype=torch.int32)
    tgt = torch.empty(n, device=DEV, dtype=torch.int64)
    count = torch.empty(1, device=DEV, dtype=torch.int32)
    nb = lib.rbm_compact_ws_bytes(n)
    ws = ops._ws("compact", nb, DEV)
    if stale:
        _stale(ws)
    L.check(lib.rbm_compact_labels(L.ptr(labels), n, L.ptr(rows), L.ptr(tgt), L.ptr(count), L.ptr(ws), nb, L.stream()), "compact")
    return rows, tgt, count


def ce_fwd(h, rows, tgt, count, w, bias, stale=False):
    lib = L.load()
    n, d = h.shape
    V1 = w.shape[0]
    full = (lambda *s: torch.full(s, float("nan"), device=DEV)) if stale else (lambda *s: torch.empty(*s, device=DEV))
    lse, loss = full(n), full(1)
    nb = lib.rbm_ce_ws_bytes(n, V1, d)
    ws = ops._ws("ce", nb, DEV)
    if stale:
        _stale(ws)
        _stale(ops._ws("compact", lib.rbm_compact_ws_bytes(n), DEV))
    L.check(lib.rbm_ce_fwd(L.ptr(h), L.ptr(rows), L.ptr(tgt), L.ptr(count), L.ptr(w), L.ptr(bias), L.ptr(lse), L.ptr(loss), n, V1, d,
                           L.ptr(ws), nb, L.stream()), "ce_fwd")
    return lse, loss


def ce_bwd(h, rows, tgt, count, w, bias, lse, dloss=1.0, stale=False):
    """dH comes back pre-zeroed (the documented contract of both callers); dW / db start as NaN under `stale`."""
    lib = L.load()
    n, d = h.shape
    V1 = w.shape[0]
    dh = torch.zeros_like(h)
    dw = torch.full_like(w, float("nan")) if stale else torch.empty_like(w)
    db = torch.full((V1,), float("nan"), device=DEV) if stale else torch.empty(V1, device=DEV)
    dl = torch.full((1,), float(dloss), device=DEV)
    nb = lib.rbm_ce_ws_bytes(n, V1, d)
    ws = ops._ws("ce", nb, DEV)
    if stale:
        _stale(ws)
        _stale(ops._ws("compact", lib.rbm_compact_ws_bytes(n), DEV))
    L.check(lib.rbm_ce_bwd(L.ptr(h), L.ptr(rows), L.ptr(tgt), L.ptr(count), L.ptr(w), L.ptr(bias), L.ptr(lse), L.ptr(dl), L.ptr(dh),
                           L.ptr(dw), L.ptr(db), n, V1, d, L.ptr(ws), nb, L.stream()), "ce_bwd")
    return dh, dw, db


def run_ce(h, labels, w, bias, stale=False):
    """One unsharded forward + backward, as ops.score_cross_entropy does it."""
    rows, tgt, count = compact(labels, stale)
    lse, loss = ce_fwd(h, rows, tgt, count, w, bias, stale)
    dh, dw, db = ce_bwd(h, rows, tgt, count, w, bias, lse, stale=stale)
    torch.cuda.synchronize()
    c = int(count.item())
    return Run(lse[:c], loss.reshape(()), dh, dw, db)


def run_sharded(h, labels, w, bias, bounds):
    """VocabParallelCEFn (dist.py) for len(bounds) - 1 virtual ranks in one process: shard s = rows [bounds[s], bounds[s+1]) of the
    output layer; per shard the forward with targets shifted by -v_begin, dist.combine_shard_lse of the stacked shard results,
    per shard the backward with the global LSE, dH summed over the shards."""
    rows, tgt, count = compact(labels)
    shards = list(zip(bounds[:-1], bounds[1:]))
    fw = [ce_fwd(h, rows, (tgt - v0).contiguous(), count, w[v0:v1], None if bias is None else bias[v0:v1]) for v0, v1 in shards]
    LSE, loss = rd.combine_shard_lse(torch.stack([f[0] for f in fw]), torch.cat([f[1] for f in fw]), count)
    LSE = LSE.contiguous()
    dh = torch.zeros_like(h)
    dws, dbs = [], []
    for v0, v1 in shards:
        dh_s, dw_s, db_s = ce_bwd(h, rows, (tgt - v0).contiguous(), count, w[v0:v1], None if bias is None else bias[v0:v1], LSE)
        dh += dh_s
        dws.append(dw_s)
        dbs.append(db_s)
    torch.cuda.synchronize()
    c = int(count.item())
    return Run(LSE[:c], loss.reshape(()), dh, torch.cat(dws), torch.cat(dbs))


# ---------------------------------------------------------------------------------------------------- inputs
def make_inputs(n, V1, d, count, seed, bias_spread=1.0, hs=0.5, ws=None):
    """h [n, d], w [V1, d], bias [V1] and labels with exactly `count` labelled rows at random positions: targets include id 1, id
    V1 - 1, an id in the last (partial) 64-row vocabulary tile and one id repeated across a third of the rows."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    ws = 1.0 / math.sqrt(d) if ws is None else ws
    h = torch.randn(n, d, device=DEV, generator=g) * hs
    w = torch.randn(V1, d, device=DEV, generator=g) * ws
    b = (torch.rand(V1, device=DEV, generator=g) * 2 - 1) * bias_spread
    labels = torch.zeros(n, dtype=torch.long, device=DEV)
    if count:
        pos = torch.randperm(n, device=DEV, generator=g)[:count]
        t = torch.randint(1, V1, (count,), device=DEV, generator=g)
        t[::3] = max(1, (V1 * 5) // 7)
        last0 = (V1 - 1) // 64 * 64
        specials = torch.tensor([1, V1 - 1, max(1, last0 + (V1 - last0) // 2)], device=DEV)[:count]
        t[:specials.numel()] = specials
        labels[pos] = t
    assert int((labels != 0).sum()) == count
    return h, labels, w, b


def check(got: Run, h, labels, w, bias, path, what="", ref=None, dloss=1.0):
    """Every output of one call against the oracle; records the error per path for the summary."""
    ref = oc.masked_ce64(h, labels, w, bias) if ref is None else ref
    c = ref.lse.shape[0]
    assert got.lse.shape[0] == c, (what, got.lse.shape, c)
    if c == 0:
        return ref
    # LSE: bound per row from the arithmetic (module docstring)
    sel = labels != 0
    ha = h[sel].abs()
    amax = torch.zeros(c, device=DEV)
    for v0 in range(0, w.shape[0], 65536):
        amax = torch.maximum(amax, (ha @ w[v0:v0 + 65536].abs().t()).amax(1))
    amax = amax.double()
    bound = 2.0 ** -20 * amax + 2.0 ** -21 * ref.lse.abs().clamp(min=1.0)
    r = float(((got.lse.double() - ref.lse).abs() / bound).max())
    WORST[path]["lse"] = max(WORST[path]["lse"], r)
    assert r <= 1.0, (what, "lse", r)
    el = abs(float(got.loss) - ref.loss)
    loss_bar = LOSS_BAR * max(abs(ref.loss), 1.0) + 2.0 ** -21 * float(amax.mean())
    WORST[path]["loss"] = max(WORST[path]["loss"], el / loss_bar)
    assert el <= loss_bar, (what, "loss", float(got.loss), ref.loss, el, loss_bar)
    for name, gv, rv in (("dH", got.dh, ref.dh), ("dW", got.dw, ref.dw), ("db", got.db, ref.db)):
        rv = rv * dloss
        e = float((gv.double() - rv).abs().max() / rv.abs().max())
        WORST[path][name] = max(WORST[path][name], e)
        assert e <= GRAD_BAR[name], (what, name, e)
    return ref


# ----------------------------------------------------------------------------------------------- dispatch matrix
# (name, n, V1, d, family)
DISPATCH = [
    ("simt_d16_DT4", 300, 1001, 16, "simt"),
    ("simt_d48_DT8", 300, 777, 48, "simt"),
    ("simt_d96_DT16", 300, 515, 96, "simt"),
    ("simt_d200_DT32", 300, 333, 200, "simt"),
    ("simt_d64_V63", 300, 63, 64, "simt"),
    ("simt_d128_V40", 300, 40, 128, "simt"),
    ("simt_d256_V17", 300, 17, 256, "simt"),
    ("tc_d32", 300, 1001, 32, "tc"),
    ("tc_d64", 300, 3417, 64, "tc"),
    ("wide_d128", 300, 2049, 128, "wide"),
    ("wide_d256", 300, 2049, 256, "wide"),
]
_ALL = SIMT + TC + WIDE
_DT = {16: 4, 48: 8, 96: 16, 200: 32, 64: 8, 128: 16, 256: 32}


def _ran(names, kernel):
    """Whether a kernel of that exact name (demangled `ns::name<...>(` or mangled `<len>name<I|E>`) is among the launches."""
    pat = re.compile(r"(?<![A-Za-z_])%s(?![a-z_])" % kernel)
    return any(pat.search(n) for n in names)


@pytest.mark.parametrize("row", DISPATCH, ids=[r[0] for r in DISPATCH])
def test_ce_dispatch_reaches_every_path(row):
    """Each row runs its family's kernels and none of another family's (a changed dispatch condition names the shape that moved);
    the SIMT rows also run the DT they are meant to (d = 16 / 48 / 96 / 200 -> DT = 4 / 8 / 16 / 32).  Each row is checked
    against the oracle as well."""
    from torch.profiler import profile, ProfilerActivity
    name, n, V1, d, fam = row
    assert path_of(V1, d) == fam
    h, labels, w, b = make_inputs(n, V1, d, n // 2, seed=len(name))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        got = run_ce(h, labels, w, b)
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    for kern in FAMILY[fam]:
        assert _ran(names, kern), (name, kern, sorted(set(names)))
    for kern in _ALL:
        if kern not in FAMILY[fam]:
            assert not _ran(names, kern), (name, kern, sorted(set(names)))
    if fam == "simt":
        dts = {int(a or b_) for nm in names for a, b_ in re.findall(r"ce_bwd_d[hw]_kernel(?:<(\d+)>|ILi(\d+)E)", nm)}
        assert dts == {_DT[d]}, (name, dts)
    check(got, h, labels, w, b, fam, name)


# ---------------------------------------------------------------------------------------------- tile and split edges
N_EDGE = 2500  # not a multiple of 1024: the last compaction block is partial


@pytest.mark.parametrize("V1", [64, 65, 127, 128, 129])
@pytest.mark.parametrize("count", [1, 127, 128, 129, N_EDGE])
@pytest.mark.parametrize("d", [96, 64, 128, 256], ids=["simt_d96", "tc_d64", "wide_d128", "wide_d256"])
def test_ce_tile_edges(d, count, V1):
    """Row counts around the 128-row tiles (and every row labelled) against vocabularies around the 64- and 128-row tiles.  On the
    split-fp16 path a small count makes the device-side split (pick_vs) create up to 64 vocabulary splits per row tile, most of
    them with an empty vocabulary range whose (-inf, 0) statistics and zero dH blocks are combined with the others."""
    h, labels, w, b = make_inputs(N_EDGE, V1, d, count, seed=count * 1000 + V1)
    check(run_ce(h, labels, w, b), h, labels, w, b, path_of(V1, d), "d=%d count=%d V1=%d" % (d, count, V1))


@pytest.mark.parametrize("V1", [4799, 4801])
@pytest.mark.parametrize("count", [47, 48, 49, 1000])
def test_ce_wide_dh_chunk_width(count, V1):
    """d = 256 streams 48-row chunks (vocabulary rows in the dH kernel, hidden rows in the dW kernel): vocabularies one either side
    of a multiple of 48 and row counts around one chunk."""
    h, labels, w, b = make_inputs(1100, V1, 256, count, seed=V1 + count)
    check(run_ce(h, labels, w, b), h, labels, w, b, "wide", "count=%d V1=%d" % (count, V1))


@pytest.mark.parametrize("d", [128, 256])
@pytest.mark.parametrize("count", [100, 200, 148 * 128, 148 * 128 + 60])
def test_ce_wide_vocabulary_splits(d, count):
    """Row-tile counts RT = 1, 2, 148, 149 on the split-fp16 path: pick_vs changes the vocabulary split count at each."""
    n = count + 37
    h, labels, w, b = make_inputs(n, 1000, d, count, seed=count + d)
    check(run_ce(h, labels, w, b), h, labels, w, b, "wide", "d=%d count=%d" % (d, count))


def test_ce_wide_past_unit_limit():
    """More than UMAX = 1184 row tiles (count > 151,552): the grid switches to one CTA per row tile with no vocabulary split."""
    n, count, V1, d = 160_000, 155_000, 300, 128
    h, labels, w, b = make_inputs(n, V1, d, count, seed=9)
    check(run_ce(h, labels, w, b), h, labels, w, b, "wide", "RT=%d" % ((count + 127) // 128))


# ---------------------------------------------------------------------------------------------- vocabulary shards
def _even(V1, S):
    return [rd.shard_range(V1, r, S)[0] for r in range(S)] + [V1]


SHARDS = [
    ("tc_d64_S2", 3000, 3417, 64, _even(3417, 2)),
    ("tc_d64_S3", 3000, 3417, 64, _even(3417, 3)),
    ("tc_d64_S8", 3000, 3417, 64, _even(3417, 8)),
    ("tc_d64_last_shard_simt", 3000, 3417, 64, [0, 1700, 3380, 3417]),
    ("wide_d128_last_shard_simt", 3000, 3000, 128, [0, 1500, 2960, 3000]),
    ("wide_d256_empty_shard", 3000, 5000, 256, [0, 2000, 3000, 5000]),
    ("simt_d48_S3", 3000, 777, 48, _even(777, 3)),
]


@pytest.mark.parametrize("row", SHARDS, ids=[r[0] for r in SHARDS])
def test_ce_vocab_shards(row):
    """VocabParallelCEFn restated for S virtual ranks on one GPU against the unsharded float64 oracle: targets outside a shard match
    no column, the backward of each shard uses the global LSE (its rows of softmax - onehot do not sum to zero).  A last shard of
    fewer than 64 rows runs the SIMT kernels while the others run a tensor path; 'empty_shard' has no labelled target in its range."""
    name, n, V1, d, bounds = row
    h, labels, w, b = make_inputs(n, V1, d, n // 2, seed=len(name) + V1)
    if "empty" in name:
        lo, hi = bounds[1], bounds[2]
        inside = (labels >= lo) & (labels < hi)
        labels[inside] = labels[inside] - lo + 1  # move them below the empty shard, keep them labelled
        assert not bool(((labels >= lo) & (labels < hi)).any())
    fams = {path_of(v1 - v0, d) for v0, v1 in zip(bounds[:-1], bounds[1:])}
    if "last_shard_simt" in name:
        assert fams == {path_of(V1, d), "simt"}
    got = run_sharded(h, labels, w, b, bounds)
    check(got, h, labels, w, b, "shard_" + "+".join(sorted(fams)), name)


def test_ce_vocab_shards_million_items():
    """BASELINE configs[3]: d = 256, V + 1 = 10^6 + 1 output rows over 8 shards of 125,001 rows (split-fp16 path on every shard)."""
    n, V1, d = 4096, 1_000_001, 256
    h, labels, w, b = make_inputs(n, V1, d, 2000, seed=3, hs=0.5, ws=0.05)
    b *= 0.1
    got = run_sharded(h, labels, w, b, _even(V1, 8))
    check(got, h, labels, w, b, "shard_wide", "configs[3] x 8 shards")


# ------------------------------------------------------------------------------------------------- bias, logit range
PATHS = [("simt_d48", 48), ("tc_d32", 32), ("tc_d64", 64), ("wide_d128", 128), ("wide_d256", 256)]


@pytest.mark.parametrize("d", [p[1] for p in PATHS], ids=[p[0] for p in PATHS])
@pytest.mark.parametrize("kind", ["none", "offset4", "spread60"])
def test_ce_bias(kind, d):
    """bias=None through the C ABI (zero bias); a contiguous bias 4 bytes past a 16-byte boundary (the scalar bias loads of the
    tensor paths); a bias spread of +-60, so softmax is nearly one-hot and the online max rescaling carries the result."""
    n, V1 = 1000, 1237
    h, labels, w, b = make_inputs(n, V1, d, 600, seed=d, bias_spread=60.0 if kind == "spread60" else 1.0)
    if kind == "none":
        b = None
    elif kind == "offset4":
        storage = torch.empty(V1 + 4, device=DEV)
        b_off = storage[1:V1 + 1]
        b_off.copy_(b)
        assert b_off.data_ptr() % 16 == 4
        b = b_off
    check(run_ce(h, labels, w, b), h, labels, w, b, path_of(V1, d), kind)


# ------------------------------------------------------------------------------- stale workspace, determinism, count 0
@pytest.mark.parametrize("d", [p[1] for p in PATHS], ids=[p[0] for p in PATHS])
@pytest.mark.parametrize("count", [1000, 333])
def test_ce_stale_workspace_and_determinism(d, count):
    """Two clean runs are bit-identical (no atomics anywhere), and a run with the cached 'ce' and 'compact' workspaces and the lse,
    dW, db outputs filled with NaN bytes before the forward and before the backward is bit-identical to them: no kernel reads an
    element it did not write.  count = n = 1000 labels every row (1000 is not a multiple of 64 or 128)."""
    n, V1 = 1000, 1237
    h, labels, w, b = make_inputs(n, V1, d, count, seed=d + count)
    a1 = run_ce(h, labels, w, b)
    a2 = run_ce(h, labels, w, b)
    s = run_ce(h, labels, w, b, stale=True)
    for nm, x, y, z in zip(("lse", "loss", "dH", "dW", "db"), a1.tensors(), a2.tensors(), s.tensors()):
        assert torch.equal(x, y), ("run-to-run", nm)
        assert torch.equal(x, z), ("stale workspace", nm, int(z.isnan().sum()))
    check(a1, h, labels, w, b, path_of(V1, d), "d=%d" % d)


@pytest.mark.parametrize("d", [p[1] for p in PATHS], ids=[p[0] for p in PATHS])
def test_ce_no_labelled_row(d):
    """No labelled row (on a stale workspace with NaN-filled outputs): the loss is NaN like F.cross_entropy's, dH, dW and db are
    exactly zero and nothing faults."""
    n, V1 = 700, 1237
    h, labels, w, b = make_inputs(n, V1, d, 0, seed=1)
    got = run_ce(h, labels, w, b, stale=True)
    assert got.lse.numel() == 0 and bool(torch.isnan(got.loss))
    for nm, t in (("dH", got.dh), ("dW", got.dw), ("db", got.db)):
        assert bool((t == 0).all()), (nm, int(t.isnan().sum()), float(t.abs().nan_to_num().max()))
