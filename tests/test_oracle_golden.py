"""Pin the CPU oracle against vectors minted from the unmodified reference
(tests/golden/make_golden.py).  CPU only."""
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import bert4rec as ob, sasrec as osr, metrics as om, optim as oo, common as oc

G = os.path.join(os.path.dirname(__file__), "golden")


def load(name):
    z = np.load(os.path.join(G, name + ".npz"), allow_pickle=False)
    return {k: z[k] for k in z.files}


def sd_of(z, prefix="sd."):
    return {k[len(prefix):]: torch.from_numpy(v).clone() for k, v in z.items() if k.startswith(prefix)}


def grads_via_autograd(sd, loss_fn):
    leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    loss = loss_fn(leaves)
    loss.backward()
    return loss.detach(), {k: (v.grad if v.grad is not None else torch.zeros_like(v)) for k, v in leaves.items()}


@pytest.mark.parametrize("name", ["bert_tiny", "bert_odd"])
def test_bert_logits_loss_grads(name):
    z = load(name)
    V, L, d, nb, h, B, seed = z["cfg"].tolist()
    sd = sd_of(z)
    assert {k: tuple(v.shape) for k, v in sd.items()} == ob.state_dict_shapes(V, L, d, nb)
    t, l = torch.from_numpy(z["tokens"]), torch.from_numpy(z["labels"])
    lg = ob.logits(sd, t, nb, h)
    np.testing.assert_allclose(lg.numpy(), z["logits"], rtol=1e-5, atol=1e-5)
    loss, grads = grads_via_autograd(sd, lambda p: ob.loss(p, t, l, nb, h))
    assert abs(loss.item() - float(z["loss"])) < 1e-5
    for k, g in grads.items():
        np.testing.assert_allclose(g.numpy(), z["grad." + k], rtol=1e-4, atol=1e-6, err_msg=k)
    # the masked-rows-only chunked restatement is the same loss
    lm = ob.loss_masked_only(sd, t, l, nb, h, chunk=16)
    assert abs(lm.item() - float(z["loss"])) < 1e-5
    # eval scoring
    ev, c = torch.from_numpy(z["eval_tokens"]), torch.from_numpy(z["candidates"])
    np.testing.assert_allclose(ob.scores_last(sd, ev, nb, h).numpy(), z["scores_last"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ob.candidate_scores(sd, ev, c, nb, h).numpy(), z["cand_scores"], rtol=1e-5, atol=1e-5)


def adam_replay(sd, loss_fn, steps, lr=1e-3):
    params = {k: v.clone().numpy() for k, v in sd.items()}
    m = {k: np.zeros_like(v) for k, v in params.items()}
    v_ = {k: np.zeros_like(v) for k, v in params.items()}
    losses = []
    for s in range(1, steps + 1):
        loss, grads = grads_via_autograd({k: torch.from_numpy(v) for k, v in params.items()}, loss_fn)
        losses.append(loss.item())
        for k in params:
            oo.adam_step(params[k], grads[k].numpy(), m[k], v_[k], s, lr)
    return losses, params


@pytest.mark.parametrize("name", ["bert_tiny"])
def test_bert_adam_steps(name):
    z = load(name)
    V, L, d, nb, h, B, seed = z["cfg"].tolist()
    t, l = torch.from_numpy(z["tokens"]), torch.from_numpy(z["labels"])
    losses, params = adam_replay(sd_of(z), lambda p: ob.loss(p, t, l, nb, h), len(z["adam_losses"]))
    np.testing.assert_allclose(losses, z["adam_losses"], rtol=2e-6)
    for k, v in sd_of(z, "sd_after.").items():
        if k.endswith("linear_layers.1.bias"):
            continue  # d loss / d b_k == 0 analytically (softmax shift invariance): Adam amplifies fp noise to +-lr
        np.testing.assert_allclose(params[k], v.numpy(), rtol=1e-4, atol=2e-6, err_msg=k)


@pytest.mark.parametrize("name", ["bert_cfg2", "bert_cfg4s"])  # configs[1] shape; configs[3] model shape (d=256, 4 blocks, h=4)
def test_bert_cfg2_shape(name):
    z = load(name)
    V, L, d, nb, h, B, seed = z["cfg"].tolist()
    sd = ob.random_state_dict(V, L, d, nb, seed=seed)
    t, l = torch.from_numpy(z["tokens"]), torch.from_numpy(z["labels"])
    loss, grads = grads_via_autograd(sd, lambda p: ob.loss_masked_only(p, t, l, nb, h))
    assert abs(loss.item() - float(z["loss"])) < 1e-4 * abs(float(z["loss"]))
    names = list(ob.state_dict_shapes(V, L, d, nb).keys())
    gn = np.array([grads[k].norm().item() for k in names], np.float32)
    np.testing.assert_allclose(gn, z["grad_norms"], rtol=1e-3, atol=1e-7)
    ev = torch.from_numpy(z["eval_tokens"])
    np.testing.assert_allclose(ob.scores_last(sd, ev, nb, h).numpy(), z["scores_last"], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("name", ["sas_tiny", "sas_odd"])
def test_sas_logits_loss_grads(name):
    z = load(name)
    V, L, d, nb, h, B, seed = z["cfg"].tolist()
    sd = sd_of(z)
    assert {k: tuple(v.shape) for k, v in sd.items()} == osr.state_dict_shapes(V, L, d, nb)
    seq, pos, neg = (torch.from_numpy(z[k]) for k in ("seq", "pos", "neg"))
    pl, nl = osr.forward(sd, seq, pos, neg, nb, h)
    np.testing.assert_allclose(pl.numpy(), z["pos_logits"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(nl.numpy(), z["neg_logits"], rtol=1e-5, atol=1e-5)
    loss, grads = grads_via_autograd(sd, lambda p: osr.loss(p, seq, pos, neg, nb, h))
    assert abs(loss.item() - float(z["loss"])) < 1e-5
    for k, g in grads.items():
        np.testing.assert_allclose(g.numpy(), z["grad." + k], rtol=1e-4, atol=2e-6, err_msg=k)
    c = torch.from_numpy(z["candidates"])
    np.testing.assert_allclose(osr.predict(sd, seq, c, nb, h).numpy(), z["cand_scores"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(osr.scores_full_catalogue(sd, seq, nb, h, chunk=16).numpy(), z["scores_full"],
                               rtol=1e-5, atol=1e-5)


def test_sas_adam_steps():
    z = load("sas_tiny")
    V, L, d, nb, h, B, seed = z["cfg"].tolist()
    seq, pos, neg = (torch.from_numpy(z[k]) for k in ("seq", "pos", "neg"))
    losses, params = adam_replay(sd_of(z), lambda p: osr.loss(p, seq, pos, neg, nb, h), len(z["adam_losses"]))
    np.testing.assert_allclose(losses, z["adam_losses"], rtol=5e-6)
    for k, v in sd_of(z, "sd_after.").items():
        a, b = params[k], v.numpy()
        if k.endswith("in_proj_bias"):  # the k-bias third has an analytically zero gradient (see BERT test)
            a, b = np.concatenate([a[:d], a[2 * d:]]), np.concatenate([b[:d], b[2 * d:]])
        np.testing.assert_allclose(a, b, rtol=1e-4, atol=2e-6, err_msg=k)


@pytest.mark.parametrize("name", ["sas_cfg1", "sas_cfg3s"])  # configs[0] shape; configs[2] model shape (d=128, h=2)
def test_sas_cfg1_shape(name):
    z = load(name)
    V, L, d, nb, h, B, seed = z["cfg"].tolist()
    sd = osr.random_state_dict(V, L, d, nb, seed=seed)
    seq, pos, neg = (torch.from_numpy(z[k]) for k in ("seq", "pos", "neg"))
    loss, grads = grads_via_autograd(sd, lambda p: osr.loss(p, seq, pos, neg, nb, h))
    assert abs(loss.item() - float(z["loss"])) < 1e-4 * abs(float(z["loss"]))
    names = list(osr.state_dict_shapes(V, L, d, nb).keys())
    gn = np.array([grads[k].norm().item() for k in names], np.float32)
    np.testing.assert_allclose(gn, z["grad_norms"], rtol=1e-3, atol=1e-7)
    np.testing.assert_allclose(osr.scores_full_catalogue(sd, seq, nb, h).numpy(), z["scores_full"], rtol=1e-4, atol=1e-4)


def test_metrics_match_reference():
    z = load("metrics")
    for tag in ("c101", "c3416", "multi"):
        scores, labels = torch.from_numpy(z[tag + ".scores"]), torch.from_numpy(z[tag + ".labels"])
        ks = [1, 5, 10, 20] if tag != "multi" else [1, 5, 10]
        m = om.recalls_ndcgs_and_mrr_for_ks(scores, labels, ks)
        keys = [str(k) for k in z[tag + ".keys"]]
        assert sorted(m.keys()) == keys
        np.testing.assert_array_equal(np.array([m[k] for k in keys], np.float64), z[tag + ".vals"])  # bit-exact
        if tag != "multi":
            # canonical rank == reference's unstable argsort when there are no ties
            np.testing.assert_array_equal(om.canonical_rank(scores)[:, :20].numpy(), z[tag + ".rank20"])
            vals, ids = om.topk_canonical(scores.numpy(), 20)
            np.testing.assert_array_equal(ids, z[tag + ".rank20"])
            pu = om.full_catalogue_metrics(ids, np.zeros(scores.shape[0], np.int64), [1, 5, 10, 20])
            ref_pu = om.recalls_ndcgs_and_mrr_for_ks(scores, labels, [1, 5, 10, 20], per_user=True)
            for k in pu:
                np.testing.assert_array_equal(pu[k], ref_pu[k].numpy(), err_msg=k)


def test_topk_merge_shard_invariant():
    rng = np.random.RandomState(0)
    U, V, k = 7, 1000, 10
    scores = rng.randn(U, V).astype(np.float32)
    scores[:, 100:110] = scores[:, 200:210]  # exact ties across shards
    ref_v, ref_i = om.topk_canonical(scores, k, id_offset=1)
    for S in (1, 2, 3, 8):
        bounds = np.linspace(0, V, S + 1).astype(int)
        parts = [om.topk_canonical(scores[:, a:b], k, id_offset=1 + a) for a, b in zip(bounds[:-1], bounds[1:])]
        v, i = om.topk_merge(np.stack([p[0] for p in parts]), np.stack([p[1] for p in parts]), k)
        np.testing.assert_array_equal(i, ref_i)
        np.testing.assert_array_equal(v, ref_v)


def test_scatter_and_adam_match_torch():
    z = load("scatter_adam")
    g = oc.embedding_grad_scatter(z["scatter.idx"], z["scatter.rows"], 53, padding_idx=0)
    np.testing.assert_array_equal(g, z["scatter.grad"])  # bit-exact, index-ordered fp32 adds
    np.testing.assert_array_equal(oc.embedding_grad_scatter_fast(z["scatter.idx"], z["scatter.rows"], 53), g)
    # the CUDA kernel's piece-tree contract: identical for rows with <= 64 contributions, rounding-level otherwise
    gc = oc.embedding_grad_scatter_chunked(z["scatter.idx"], z["scatter.rows"], 53)
    short = np.bincount(z["scatter.idx"], minlength=53) <= 64
    np.testing.assert_array_equal(gc[short], g[short])
    np.testing.assert_allclose(gc, g, rtol=1e-5, atol=1e-5)
    p = z["adam.p0"].copy()
    m, v = np.zeros_like(p), np.zeros_like(p)
    for s in range(4):
        oo.adam_step(p, z["adam.grads"][s], m, v, s + 1, 1e-3)
        np.testing.assert_allclose(p, z["adam.ps"][s], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(m, z["adam.m"], rtol=1e-5, atol=1e-8)
    np.testing.assert_allclose(v, z["adam.v"], rtol=1e-6, atol=1e-12)


def test_injected_dropout_masks():
    """Injected-mask mode == torch's dropout formula (x * keep / (1-p))."""
    x = torch.randn(3, 5)
    keep = (torch.rand(3, 5) > 0.3).to(torch.uint8)
    d = oc.DropoutPlan(training=True, masks={4: keep})
    np.testing.assert_allclose(d(x, 0.3, 4).numpy(), (x * keep / 0.7).numpy(), rtol=1e-6)
    assert oc.DropoutPlan(training=False)(x, 0.3, 4) is x


# ------------------------------------------------------------------------------------ batch construction
def test_philox_known_answers():
    """Philox4x32-10 known-answer vectors of the Random123 distribution (kat_vectors)."""
    from oracle.batches import philox4x32_10
    assert philox4x32_10((0, 0, 0, 0), (0, 0)) == (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)
    assert philox4x32_10((0xffffffff,) * 4, (0xffffffff, 0xffffffff)) == (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)
    assert philox4x32_10((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0)) == (
        0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)
    from oracle.batches import philox4x32  # the same vectors as one array call
    cs = np.array([[0, 0xffffffff, 0x243f6a88], [0, 0xffffffff, 0x85a308d3], [0, 0xffffffff, 0x13198a2e], [0, 0xffffffff, 0x03707344]])
    got = philox4x32(list(cs), (0xa4093822, 0x299f31d0), 10)
    assert [int(w[2]) for w in got] == [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


@pytest.mark.parametrize("L", [1, 7, 16, 17, 40])
def test_dropout_masks_restate_the_per_element_rule(L):
    """The vectorised masks of oracle/common.py against a per-element transcription of the scalar rules of csrc/common.cuh
    (rbm_drop4, rbm_attn_keep): seed and site with their high 32 bits set."""
    from oracle.batches import philox4x32
    seed, site, p = (0xA5A5 << 32) | 77, (3 << 32) | 9, 0.3

    def r7(call):
        return [int(w) for w in philox4x32((call & 0xFFFFFFFF, call >> 32, site & 0xFFFFFFFF, site >> 32), (seed & 0xFFFFFFFF, seed >> 32), 7)]

    thr = int(float(np.float32(p)) * 2 ** 32)
    n = 4 * L + 3
    assert oc.keep_mask(n, p, seed, site).tolist() == [r7(e // 4)[e % 4] >= thr for e in range(n)]
    thr16 = int(float(np.float32(p)) * 65536 + 0.5)
    BH = 3
    got = oc.attn_keep_mask(BH, L, p, seed, site)
    for bh in range(BH):
        for i in range(L):
            for j in range(L):
                r = r7((((bh * 16 + (i >> 4)) * 8 + (i & 7)) * 4 + ((j & 7) >> 1)) * 16 + (j >> 4))
                f = ((i >> 3) & 1) * 4 + (j & 1) * 2 + ((j >> 3) & 1)
                w = r[f >> 1]
                assert bool(got[bh * L + i, j]) == (((w >> 16) if f & 1 else (w & 0xFFFF)) >= thr16), (bh, i, j)


def _histories(z):
    ptr, items = z["hist_ptr"], z["hist_items"]
    return [items[ptr[u]:ptr[u + 1]].tolist() for u in range(len(ptr) - 1)]


@pytest.mark.parametrize("tag,L", [("bert_L8", 8), ("bert_L16_all", 16), ("bert_L8_none", 8)])
def test_bert_cloze_batch_vs_reference_dataset(tag, L):
    """oracle.batches.bert_cloze_batch == the reference's BertTrainDataset driven by the same random numbers."""
    from oracle import batches as obt
    z = load("batches")
    V = int(z["num_items"])
    t, l = obt.bert_cloze_batch(_histories(z), z[tag + ".users"].tolist(), L, float(z[tag + ".mask_prob"]), V + 1, V,
                                int(z["seed"]), int(z["site"]))
    np.testing.assert_array_equal(t, z[tag + ".tokens"])
    np.testing.assert_array_equal(l, z[tag + ".labels"])


@pytest.mark.parametrize("tag,L", [("sas_L8", 8), ("sas_L50", 50)])
def test_sas_train_batch_vs_reference_sampler(tag, L):
    """oracle.batches.sas_train_batch == the reference's sample_function driven by the same random numbers."""
    from oracle import batches as obt
    z = load("batches")
    s, p, n = obt.sas_train_batch(_histories(z), z[tag + ".users"].tolist(), L, int(z["num_items"]), int(z["seed"]), int(z["site"]))
    np.testing.assert_array_equal(s, z[tag + ".seq"])
    np.testing.assert_array_equal(p, z[tag + ".pos"])
    np.testing.assert_array_equal(n, z[tag + ".neg"])


# ------------------------------------------------------------------------------------ evaluation negatives / batches
def _split(z, name):
    ptr, items = z[name + "_ptr"], z[name + "_items"]
    return [items[ptr[u]:ptr[u + 1]].tolist() for u in range(len(ptr) - 1)]


@pytest.mark.parametrize("code", ["random", "popular"])
def test_negative_samples_vs_reference_sampler(code):
    """oracle.batches.negative_samples == Random / PopularNegativeSampler.generate_negative_samples of the reference driven
    by the same random numbers (tests/golden/eval_batches.npz)."""
    from oracle import batches as obt
    z = load("eval_batches")
    tr, va, te = _split(z, "train"), _split(z, "val"), _split(z, "test")
    seen = [sorted(set(tr[u]) | set(va[u]) | set(te[u])) for u in range(len(tr))]
    out = obt.negative_samples(seen, int(z["num_items"]), int(z["sample_size"]), int(z["seed"]), int(z["site"]),
                               pop_counts=z["pop_counts"].tolist() if code == "popular" else None)
    np.testing.assert_array_equal(out, z["neg_" + code])
    for u in range(len(tr)):  # what the samplers promise: distinct, unseen, in range
        row = out[u].tolist()
        assert len(set(row)) == len(row) and not (set(row) & set(seen[u])) and min(row) >= 1 and max(row) <= int(z["num_items"])
    # a sub-range of users is the same rows (the counter is the user id, not the row)
    part = obt.negative_samples(seen, int(z["num_items"]), int(z["sample_size"]), int(z["seed"]), int(z["site"]),
                                pop_counts=z["pop_counts"].tolist() if code == "popular" else None, user_begin=3, num_users=4)
    np.testing.assert_array_equal(part, out[3:7])


@pytest.mark.parametrize("model,L", [("bert", 8), ("bert", 16), ("sas", 8), ("sas", 16)])
def test_eval_batch_vs_reference_dataset(model, L):
    """oracle.batches.eval_batch == BertEvalDataset / SASEvalDataset.__getitem__ of the reference."""
    from oracle import batches as obt
    z = load("eval_batches")
    tr, va = _split(z, "train"), _split(z, "val")
    V = int(z["num_items"])
    users = list(range(len(tr)))
    s, c, l = obt.eval_batch(tr, [v[0] for v in va], z["neg_random"], users, L, V + 1 if model == "bert" else -1)
    np.testing.assert_array_equal(s, z["%s_L%d.seq" % (model, L)])
    np.testing.assert_array_equal(c, z["%s_L%d.cand" % (model, L)])
    np.testing.assert_array_equal(l, z["%s_L%d.labels" % (model, L)])


def test_negative_samples_unfillable_row_ends_in_minus_one():
    from oracle import batches as obt
    out = obt.negative_samples([[1, 2, 3, 4], [2]], 5, 2, 9, 1 << 41)
    assert out[0].tolist()[0] == 5 and out[0].tolist()[1] == -1 and (out[1] > 0).all()


# ------------------------------------------------------------------------------------ data_partition (SURVEY 8(f) #4)
@pytest.mark.parametrize("L,prop,tag", [(8, 0.3, "L8_p03"), (50, 0.3, "L50_p03"), (50, -1.0, "L50_pm10"), (200, 0.3, "L200_p03")])
def test_data_partition_vs_reference(tmp_path, L, prop, tag):
    """The vectorised text parser + sliding-window split == the reference's data_partition on the same file
    (tests/golden/partition.npz: interleaved users, histories shorter than 3, equal to / just above max_len, many windows)."""
    from rbm_b200.dataloaders import data_partition
    z = load("partition")
    f = tmp_path / "interactions.txt"
    f.write_bytes(z["text"].tobytes())
    tr, va, te, n, V = data_partition(str(f), L, prop)
    assert n == int(z[tag + ".n"]) == len(tr) == len(va) == len(te) and V == int(z[tag + ".V"])
    ptr = z[tag + ".train_ptr"]
    assert [len(r) for r in tr] == np.diff(ptr).tolist()
    np.testing.assert_array_equal(np.array([i for r in tr for i in r], np.int64), z[tag + ".train"])
    np.testing.assert_array_equal(np.array([r[0] for r in va], np.int64), z[tag + ".valid"])
    np.testing.assert_array_equal(np.array([r[0] for r in te], np.int64), z[tag + ".test"])


# --------------------------------------------------------------------------------- masked cross-entropy in float64
def _ce_inputs(n, V1, d, seed, frac=0.6):
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(n, d, generator=g, dtype=torch.float64)
    w = torch.randn(V1, d, generator=g, dtype=torch.float64) * 0.4
    b = torch.randn(V1, generator=g, dtype=torch.float64)
    labels = torch.where(torch.rand(n, generator=g) < frac, torch.randint(1, V1, (n,), generator=g), torch.zeros(n, dtype=torch.long))
    return h, labels, w, b


@pytest.mark.parametrize("n,V1,d,frac,bias", [(23, 17, 8, 0.6, True), (40, 101, 16, 0.3, False), (9, 5, 4, 1.0, True), (12, 30, 8, 0.0, True)])
def test_masked_ce64_equals_torch(n, V1, d, frac, bias):
    """oc.masked_ce64 is F.cross_entropy(h.w^T + b, labels, ignore_index=0) in float64: loss, dH, dW, db (chunked over a
    vocabulary that is not a multiple of the chunk); bias=None is a zero bias; no labelled row gives a NaN loss and zero
    gradients, as torch does."""
    h, labels, w, b = _ce_inputs(n, V1, d, n)
    if not bias:
        b = torch.zeros_like(b)
    leaves = [t.clone().requires_grad_(True) for t in (h, w, b)]
    ref = F.cross_entropy(F.linear(*leaves), labels, ignore_index=0)
    ref.backward()
    got = oc.masked_ce64(h, labels, w, b if bias else None, chunk=7)
    sel = labels != 0
    assert got.lse.shape == (int(sel.sum()),)
    if not bool(sel.any()):
        assert math.isnan(got.loss) and math.isnan(ref.item())
        assert not got.dh.any() and not got.dw.any() and not got.db.any()
        assert not leaves[0].grad.any() and not leaves[1].grad.any()
        return
    torch.testing.assert_close(got.lse, torch.logsumexp(F.linear(h, w, b)[sel], 1), rtol=1e-13, atol=1e-13)
    assert abs(got.loss - ref.item()) < 1e-13 * abs(ref.item())
    torch.testing.assert_close(got.dh, leaves[0].grad, rtol=1e-12, atol=1e-14)
    torch.testing.assert_close(got.dw, leaves[1].grad, rtol=1e-12, atol=1e-14)
    torch.testing.assert_close(got.db, leaves[2].grad, rtol=1e-12, atol=1e-14)

@pytest.mark.parametrize("bounds", [[0, 37], [0, 20, 37], [0, 13, 26, 37], [0, 5, 10, 15, 20, 25, 30, 35, 37],
                                    [0, 30, 35, 36, 37], [0, 1, 36, 37]], ids=lambda b: "S%d_%s" % (len(b) - 1, "_".join(map(str, b))))
def test_masked_ce64_vocab_shards_combine(bounds):
    """The vocabulary-parallel loss restated with the oracle: per shard [v_begin, v_end) the forward with labels shifted by
    -v_begin (a target outside the shard contributes no column), dist.combine_shard_lse of the shard log-sum-exps and losses,
    per shard the backward with the global log-sum-exp, dH summed over the shards.  It reproduces the unsharded log-sum-exp,
    loss, dW, db and dH for 1, 2, 3 and 8 shards, uneven last shards and one-row shards."""
    from rbm_b200 import dist as rd
    n, V1, d = 60, bounds[-1], 8
    h, labels, w, b = _ce_inputs(n, V1, d, 7)
    labels[3], labels[4] = V1 - 1, 1  # the last and first scored ids
    full = oc.masked_ce64(h, labels, w, b)
    shards = [oc.masked_ce64(h, labels, w[v0:v1], b[v0:v1], v_begin=v0) for v0, v1 in zip(bounds[:-1], bounds[1:])]
    count = torch.tensor([full.lse.shape[0]], dtype=torch.int32)
    LSE, loss = rd.combine_shard_lse(torch.stack([s.lse for s in shards]), torch.tensor([s.loss for s in shards]), count)
    torch.testing.assert_close(LSE.double(), full.lse, rtol=1e-6, atol=1e-6)
    assert abs(loss.item() - full.loss) < 1e-6 * abs(full.loss)
    if len(bounds) > 2:  # a shard's own rows of softmax - onehot do not sum to zero: the global LSE matters
        assert (shards[0].lse - full.lse).abs().max() > 0.1
    back = [oc.masked_ce64(h, labels, w[v0:v1], b[v0:v1], v_begin=v0, lse=LSE) for v0, v1 in zip(bounds[:-1], bounds[1:])]
    torch.testing.assert_close(torch.cat([s.dw for s in back]), full.dw, rtol=1e-5, atol=1e-8)
    torch.testing.assert_close(torch.cat([s.db for s in back]), full.db, rtol=1e-5, atol=1e-8)
    torch.testing.assert_close(sum(s.dh for s in back), full.dh, rtol=1e-5, atol=1e-8)
