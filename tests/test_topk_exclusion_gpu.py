"""Full-catalogue top-k that leaves out each user's seen items (``rbm_score_topk_excl``, ``ops.score_topk(exclude=...)``): every
kernel path against the canonical top-k of the remaining items, the models, the sharded path, and the opt-in full-catalogue
protocol of the loaders and trainers (``args.full_catalogue_eval``)."""
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import metrics as om

DEV = "cuda"


def topk_canonical_excluding(scores, exclude, k, id_offset=0):
    """Canonical (score desc, id asc) top-k per row of ``scores`` [U, C] (ids = column + id_offset) after the ids of row u of
    ``exclude`` are removed; ids outside [id_offset, id_offset + C) remove nothing.  Fewer than k left: (-inf, -1) padding --
    ``oracle.metrics.topk_canonical`` on the remaining columns."""
    scores = np.asarray(scores, np.float32)
    U, C = scores.shape
    vals = np.full((U, k), -np.inf, np.float32)
    ids = np.full((U, k), -1, np.int64)
    for u in range(U):
        cols = np.asarray(exclude[u], np.int64) - id_offset
        keep = np.ones(C, bool)
        keep[cols[(cols >= 0) & (cols < C)]] = False
        idx = np.nonzero(keep)[0]
        if idx.size == 0:
            continue
        v, i = om.topk_canonical(scores[u:u + 1, idx], k)
        n = min(k, idx.size)
        vals[u, :n], ids[u, :n] = v[0, :n], idx[i[0, :n]] + id_offset
    return vals, ids


# ------------------------------------------------------------------------------------------------ CPU: the oracle helper
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_oracle_excluding_matches_brute_force(seed):
    """topk_canonical_excluding against a plain python loop over (score, id) pairs: ties, duplicates, padding, other ids."""
    rng = np.random.RandomState(seed)
    U, C, k, off = 7, 40, 10, 3
    scores = np.round(rng.randn(U, C), 1).astype(np.float32)  # plenty of ties
    exclude = [list(rng.randint(-2, C + 8, size=rng.randint(0, C + 5))) for _ in range(U)]
    exclude[0] = list(range(off, off + C - 4))  # four items left: six padding slots
    exclude[1] = []
    vals, ids = topk_canonical_excluding(scores, exclude, k, id_offset=off)
    for u in range(U):
        ex = set(int(e) for e in exclude[u])
        pairs = sorted(((-float(scores[u, c]), c + off) for c in range(C) if c + off not in ex))[:k]
        pairs += [(np.inf, -1)] * (k - len(pairs))
        assert ids[u].tolist() == [p[1] for p in pairs]
        assert vals[u].tolist() == [-p[0] for p in pairs]


# ------------------------------------------------------------------------------------------------ GPU: kernels
@pytest.mark.gpu
def test_score_topk_rejects_bad_exclude():
    """Device, dtype and shape of ``exclude`` are checked against the users before anything runs."""
    from rbm_b200 import ops
    f, t = torch.zeros(4, 16, device=DEV), torch.zeros(10, 16, device=DEV)
    for bad in (torch.zeros(4, 3, dtype=torch.int64), torch.zeros(4, 3, dtype=torch.int32, device=DEV),
                torch.zeros(5, 3, dtype=torch.int64, device=DEV), torch.zeros(4, dtype=torch.int64, device=DEV)):
        with pytest.raises(RuntimeError):
            ops.score_topk(f, t, None, 1, 10, 5, exclude=bad)


def _exclusion_rows(sc, U, V, rng, n_rand=20):
    """Rows in output-id space (items 1..V): each user's unfiltered top-32 plus random items, shuffled, with duplicates,
    0 / -1 padding and out-of-range ids; user 0 has an all-padding row."""
    top32 = np.argsort(-sc, axis=1, kind="stable")[:, :32] + 1
    rows = []
    for u in range(U):
        r = np.concatenate([top32[u], rng.randint(1, V + 1, size=n_rand), top32[u, :3], [0, -1, V + 1, V + 7, -5]])
        if u == 0:
            r = np.zeros_like(r)
        rng.shuffle(r)
        rows.append(r)
    return np.stack(rows).astype(np.int64)


# path of each shape (rbm_score_topk's dispatch): V < 8192 or d % 32 != 0 -> fp32 scan (SIMT); k > 10 -> fp32 scan;
# otherwise tcgen05, kind::tf32 for d = 32 and range-scaled fp16 for d % 64 == 0
PATHS = [("simt_d16", 40, 3000, 16, 10), ("tc_tf32_d32", 70, 9000, 32, 10), ("tc_f16_d64", 300, 20000, 64, 10),
         ("tc_f16_d128", 130, 12101, 128, 10), ("tc_f16_d256", 64, 9000, 256, 10), ("scan_k16", 33, 9000, 64, 16)]


@pytest.mark.gpu
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("path,U,V,d,k", PATHS)
def test_score_topk_excluding_every_path(path, U, V, d, k, bias):
    """ids AND scores equal the canonical top-k of the fp32 scores (sequential FMA) over the items left after exclusion, on
    every row, with adversarial rows (each user's own top-32 excluded, so every candidate list would otherwise fill with
    excluded ids), unsorted rows, duplicates, padding, out-of-range ids and an empty row -- and again with every user forced
    through the exact re-scan (stage 3, which must filter with the user of each listed slot)."""
    from rbm_b200 import ops
    torch.manual_seed(U + V + d)
    f, table = torch.randn(U, d, device=DEV), torch.randn(V + 1, d, device=DEV)
    b = torch.randn(V + 1, device=DEV) if bias else None
    sc = om.scores_fp32_sequential(f, table[1:], b[1:] if bias else None).cpu().numpy()
    ex = _exclusion_rows(sc, U, V, np.random.RandomState(d))
    ref_v, ref_i = topk_canonical_excluding(sc, ex, k, id_offset=1)
    for eps in (None, "1e9"):
        if eps:
            os.environ["RBM_TOPK_EPS"] = eps
        try:
            vals, ids = ops.score_topk(f, table, b, 1, V + 1, k, exclude=torch.from_numpy(ex).to(DEV))
        finally:
            os.environ.pop("RBM_TOPK_EPS", None)
        np.testing.assert_array_equal(ids.cpu().numpy(), ref_i, err_msg="%s eps=%s" % (path, eps))
        np.testing.assert_array_equal(vals.cpu().numpy(), ref_v, err_msg="%s eps=%s" % (path, eps))


@pytest.mark.gpu
@pytest.mark.parametrize("V,d", [(12, 16), (8200, 64)])
def test_score_topk_excluding_leaves_fewer_than_k(V, d):
    """A user left with fewer than k items gets trailing (-inf, -1): a 12-item range (fp32 scan) and an 8200-item range on the
    tcgen05 path where one user excludes all but 4 items (its lists cannot fill: the certificate sends it to the re-scan)."""
    from rbm_b200 import ops
    torch.manual_seed(V)
    U, k = 5, 10
    f, table = torch.randn(U, d, device=DEV), torch.randn(V + 1, d, device=DEV)
    rng = np.random.RandomState(V)
    keep = rng.choice(np.arange(1, V + 1), size=4, replace=False)
    n = V - 4
    ex = np.zeros((U, n), np.int64)
    ex[0] = np.setdiff1d(np.arange(1, V + 1), keep)
    ex[1, : V // 2] = rng.permutation(np.arange(1, V + 1))[: V // 2]
    sc = om.scores_fp32_sequential(f, table[1:]).cpu().numpy()
    ref_v, ref_i = topk_canonical_excluding(sc, ex, k, id_offset=1)
    assert (ref_i[0, 4:] == -1).all() and np.isin(ref_i[0, :4], keep).all()
    vals, ids = ops.score_topk(f, table, None, 1, V + 1, k, exclude=torch.from_numpy(ex).to(DEV))
    np.testing.assert_array_equal(ids.cpu().numpy(), ref_i)
    np.testing.assert_array_equal(vals.cpu().numpy(), ref_v)


@pytest.mark.gpu
@pytest.mark.parametrize("U,V,d", [(40, 3000, 16), (300, 20000, 64)])
def test_score_topk_no_exclusion_is_bit_identical(U, V, d):
    """exclude=None, an all-zero exclude and an empty [U, 0] exclude give exactly today's result (fp32 scan and tcgen05 shapes)."""
    from rbm_b200 import ops
    torch.manual_seed(U)
    f, table, b = torch.randn(U, d, device=DEV), torch.randn(V + 1, d, device=DEV), torch.randn(V + 1, device=DEV)
    v0, i0 = ops.score_topk(f, table, b, 1, V + 1, 10)
    for ex in (None, torch.zeros(U, 37, dtype=torch.int64, device=DEV), torch.zeros(U, 0, dtype=torch.int64, device=DEV)):
        v1, i1 = ops.score_topk(f, table, b, 1, V + 1, 10, exclude=ex)
        assert torch.equal(i1, i0) and torch.equal(v1, v0)


def _shard_merge(f, table, b, V, k, ex):
    """Two calls on the two halves of the item rows (each a table of its own, ids through id_offset), merged."""
    from rbm_b200 import ops
    half = 1 + V // 2
    va, ia = ops.score_topk(f, table[1:half], b[1:half], 0, half - 1, k, id_offset=1, exclude=ex)
    vb, ib = ops.score_topk(f, table[half:], b[half:], 0, V + 1 - half, k, id_offset=half, exclude=ex)
    return ops.topk_merge(torch.stack([va, vb]), torch.stack([ia, ib]))


@pytest.mark.gpu
def test_score_topk_excluding_shard_invariance():
    """Two half-range calls with id_offset (each filtering the same global-id rows: the other half's ids never match), merged
    by topk_merge, equal one full call -- ids and scores."""
    from rbm_b200 import ops
    torch.manual_seed(3)
    U, V, d, k = 200, 40000, 64, 10
    f, table, b = torch.randn(U, d, device=DEV), torch.randn(V + 1, d, device=DEV), torch.randn(V + 1, device=DEV)
    sc = om.scores_fp32_sequential(f, table[1:], b[1:]).cpu().numpy()
    ex = torch.from_numpy(_exclusion_rows(sc, U, V, np.random.RandomState(1))).to(DEV)
    vals, ids = ops.score_topk(f, table, b, 1, V + 1, k, exclude=ex)
    mv, mi = _shard_merge(f, table, b, V, k, ex)
    assert torch.equal(mi, ids) and torch.equal(mv, vals)


@pytest.mark.gpu
def test_score_topk_excluding_million_items():
    """10^6 items, d = 64, bias: each user excludes its own unfiltered top-32 plus 18 random items.  ids and scores equal the
    canonical top-k of the fp32 scores over the rest on a sample of users, and two merged half-range calls equal one call
    (every row)."""
    from rbm_b200 import ops
    torch.manual_seed(11)
    U, V, d, k, n = 1024, 1_000_003, 64, 10, 128
    f, table, b = torch.randn(U, d, device=DEV), torch.randn(V + 1, d, device=DEV), torch.randn(V + 1, device=DEV)
    exact = f @ table[1:].t() + b[1:]  # only to pick each user's top-32 (fp32 rounding order does not matter here)
    top = torch.topk(exact, 32, dim=1).indices + 1
    del exact
    ex = torch.cat([top, torch.randint(1, V + 1, (U, 18), device=DEV)], 1)
    ex = ex[:, torch.randperm(ex.shape[1], device=DEV)].contiguous()
    vals, ids = ops.score_topk(f, table, b, 1, V + 1, k, exclude=ex)
    sc32 = om.scores_fp32_sequential(f[:n], table[1:], b[1:])
    sc32.scatter_(1, ex[:n] - 1, float("-inf"))
    rv, ri = torch.topk(sc32, k + 1, dim=1)
    assert bool((rv[:, :-1] > rv[:, 1:]).all())  # no exact ties among the top scores of random data: topk == canonical order
    assert torch.equal(ids[:n], ri[:, :k] + 1) and torch.equal(vals[:n], rv[:, :k])
    assert not bool((ids.unsqueeze(2) == ex.unsqueeze(1)).any())  # no user is offered one of its own excluded items
    mv, mi = _shard_merge(f, table, b, V, k, ex)
    assert torch.equal(mi, ids) and torch.equal(mv, vals)


# ------------------------------------------------------------------------------------------------ GPU: models
def _bert_args(V, Ln, d, nb, h, seed=0):
    return SimpleNamespace(model_code="bert", num_items=V, max_len=Ln, device=DEV, model_init_seed=seed, bert_num_blocks=nb,
                           bert_num_heads=h, bert_hidden_units=d, bert_dropout=0.0, bert_hidden_dropout=0.0)


def _sas_args(V, Ln, d, nb, h):
    return SimpleNamespace(model_code="sas", num_items=V, max_len=Ln, device=DEV, sas_hidden_units=d, sas_num_blocks=nb, sas_heads=h,
                           sas_dropout=0.0)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bert", "sas"])
def test_models_full_catalogue_topk_excluding(kind):
    """BERT4Rec / SASRec ``full_catalogue_topk(..., exclude=...)`` against the oracle on the model's own last hidden rows
    (tcgen05 path: 9000 items, d = 64); SASRec with ``exclude=log_seqs`` (everything that is not in the input)."""
    import rbm_b200
    V, Ln, d, B = 9000, 20, 64, 48
    rng = np.random.RandomState(4)
    seq = rng.randint(1, V + 1, size=(B, Ln)).astype(np.int64)
    seq[:, :3] = 0
    if kind == "bert":
        model = rbm_b200.model_factory(_bert_args(V, Ln, d, 2, 2, seed=2)).to(DEV).eval()
        seq[:, -1] = V + 1  # [MASK] at the last position
        ex = np.where(seq == V + 1, 0, seq)
        W, bias = model.out.weight, model.out.bias
    else:
        model = rbm_b200.model_factory(_sas_args(V, Ln, d, 2, 1)).to(DEV).eval()
        ex = seq
        W, bias = model.sas.item_emb.weight, None
    with torch.no_grad():
        h = model.last_hidden(torch.from_numpy(seq).to(DEV))
        vals, ids = model.full_catalogue_topk(torch.from_numpy(seq), 10, exclude=torch.from_numpy(ex) if kind == "bert" else seq)
        sc = om.scores_fp32_sequential(h, W[1:V + 1], bias[1:V + 1] if bias is not None else None).cpu().numpy()
    ref_v, ref_i = topk_canonical_excluding(sc, ex, 10, id_offset=1)
    np.testing.assert_array_equal(ids.cpu().numpy(), ref_i)
    np.testing.assert_array_equal(vals.cpu().numpy(), ref_v)


# ------------------------------------------------------------------------------------------------ GPU: loaders and trainers
def _toy_args(kind, tmp_path, **over):
    rs = np.random.RandomState(8)
    V, Ln = 90, 12
    lines = ["%d %d" % (u, i) for u in range(1, 41) for i in rs.randint(1, V + 1, size=rs.randint(3, 30))]
    f = tmp_path / "toy.txt"
    f.write_text("\n".join(lines) + "\n")
    common = dict(model_code=kind, data_path=str(f), data_name="toy.txt", max_len=Ln, prop_sliding_window=0.3, device=DEV,
                  load_processed_dataset=False, dataloader_random_seed=3, worker_number=0, train_batch_size=16, val_batch_size=8,
                  test_batch_size=8, test_negative_sampler_code="random", test_negative_sample_size=20,
                  test_negative_sampling_seed=98765, bert_mask_prob=0.3, optimizer="Adam", lr=1e-3, weight_decay=0, momentum=None,
                  decay_step=10, gamma=1.0, num_epochs=1, metric_ks=[1, 5, 10], best_metric="NDCG@10", resume_path=None, l2_emb=0.0)
    extra = vars(_bert_args(0, Ln, 16, 1, 2, seed=1)) if kind == "bert" else vars(_sas_args(0, Ln, 16, 1, 1))
    return SimpleNamespace(**{**extra, **common, **over})


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["bert", "sas"])
def test_trainer_full_catalogue_protocol(kind, tmp_path):
    """``full_catalogue_eval=True``: val / test batches are (seq, answers, exclude) with exclude = the history the loader holds
    (train; train + val) minus the answer; ``validate()`` returns the oracle's per-batch means (full-catalogue top-10 of the
    rest, HR / NDCG / MRR) to 1e-6.  Flag off (False or absent): the sampled protocol's batches and metrics, unchanged."""
    import rbm_b200
    from rbm_b200.dataloaders import data_partition
    args = _toy_args(kind, tmp_path, full_catalogue_eval=True)
    train, val, test = rbm_b200.dataloader_factory(args)
    tr, va, te, n, itemnum = data_partition(args.data_path, args.max_len, 0.3)
    off = _toy_args(kind, tmp_path)
    _, val_off, test_off = rbm_b200.dataloader_factory(off)
    for loader, loader_off, hist, ans in ((val, val_off, tr, [v[0] for v in va]),
                                          (test, test_off, [tr[u] + va[u] for u in range(n)], [t[0] for t in te])):
        u0 = 0
        for (seq, answers, ex), (seq_off, _, _) in zip(loader, loader_off):
            B = seq.shape[0]
            assert answers.shape == (B,) and ex.dim() == 2 and ex.shape[0] == B and ex.dtype == torch.int64
            assert torch.equal(seq, seq_off)
            assert answers.tolist() == ans[u0:u0 + B]
            for r, u in enumerate(range(u0, u0 + B)):
                row = ex[r].tolist()
                assert ans[u] not in row
                assert sorted(x for x in row if x != 0) == sorted(x for x in hist[u] if x != ans[u])
            assert ex.shape[1] == max(len(hist[u]) for u in range(u0, u0 + B))
            u0 += B
        assert u0 == n
    model = rbm_b200.model_factory(args)
    trainer = rbm_b200.trainer_factory(args, model, train, val, test, None)
    got = trainer.validate(0, 0)
    ks = args.metric_ks
    sums = {}
    model.eval()
    W = model.out.weight if kind == "bert" else model.sas.item_emb.weight
    bias = model.out.bias if kind == "bert" else None
    with torch.no_grad():
        for seq, answers, ex in val:
            h = model.last_hidden(seq)
            sc = om.scores_fp32_sequential(h, W[1:itemnum + 1], bias[1:itemnum + 1] if bias is not None else None).cpu().numpy()
            _, ids = topk_canonical_excluding(sc, ex.cpu().numpy(), max(ks), id_offset=1)
            for name, v in om.full_catalogue_metrics(ids, answers.cpu().numpy(), ks).items():
                sums.setdefault(name, []).append(float(np.mean(v, dtype=np.float64)))
    ref = {name: float(np.mean(v)) for name, v in sums.items()}
    assert set(got) == set(ref)
    for name in ref:
        assert abs(got[name] - ref[name]) <= 1e-6, (name, got[name], ref[name])
    # flag off: the sampled 1 + N protocol, same batches and metrics whether the field is False or absent
    args_off = _toy_args(kind, tmp_path, full_catalogue_eval=False)
    _, val_f, _ = rbm_b200.dataloader_factory(args_off)
    trainer_off = rbm_b200.trainer_factory(args_off, model, train, val_f, None, None)
    trainer_abs = rbm_b200.trainer_factory(off, model, train, val_off, None, None)
    model.eval()
    with torch.no_grad():
        for b1, b2 in zip(val_f, val_off):
            assert len(b1) == 3 and all(torch.equal(x, y) for x, y in zip(b1, b2))
            assert b1[1].shape[1] == 21
            assert trainer_off.calculate_metrics(b1) == trainer_abs.calculate_metrics(b2)
    # cut-offs above 32 are refused, as on the sampled path
    args.metric_ks = [40]
    trainer_big = rbm_b200.trainer_factory(args, model, train, val, test, None)
    with pytest.raises(RuntimeError):
        trainer_big.calculate_metrics(next(iter(val)))


# ------------------------------------------------------------------------------------------------ GPU: two ranks
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        import rbm_b200
        from rbm_b200.dist import shard_bert_model, sharded_full_catalogue_topk
        dev = "cuda:%d" % rank
        V, Ln, d, B = 9000, 24, 64, 6
        args = SimpleNamespace(**{**vars(_bert_args(V, Ln, d, 2, 2, seed=0)), "device": dev})
        rs = np.random.RandomState(3)
        tok = rs.randint(1, V + 1, size=(world * B, Ln)).astype(np.int64)
        tok[:, :2] = 0
        tok[:, -1] = V + 1
        hist = np.where(tok == V + 1, 0, tok)
        widths = [Ln, Ln // 2]  # ranks pass exclusion rows of different widths: padded to the widest before the gather
        sl = slice(rank * B, (rank + 1) * B)
        full = rbm_b200.model_factory(args).to(dev).eval()
        sh = shard_bert_model(rbm_b200.model_factory(args).to(dev)).eval()
        ex_rank = torch.from_numpy(np.ascontiguousarray(hist[sl][:, -widths[rank]:]))
        ex_full = torch.zeros(world * B, Ln, dtype=torch.int64)
        for r in range(world):
            ex_full[r * B:(r + 1) * B, :widths[r]] = torch.from_numpy(hist[r * B:(r + 1) * B, -widths[r]:])
        with torch.no_grad():
            fv, fi = full.full_catalogue_topk(torch.from_numpy(tok), 10, exclude=ex_full)
            sv, si = sh.full_catalogue_topk(torch.from_numpy(tok[sl]), 10, exclude=ex_rank)
            assert not bool((si.unsqueeze(2) == ex_rank.to(dev).unsqueeze(1)).any())
            assert torch.equal(si, fi[sl]), (si, fi[sl])
            assert torch.allclose(sv, fv[sl], rtol=1e-6, atol=1e-6)
            # replicated users, vocabulary-sharded table: the exclusion rows pass straight through to every shard
            hl = full.last_hidden(torch.from_numpy(tok).to(dev))
            exd = ex_full.to(dev)
            v1, i1 = rbm_b200.ops.score_topk(hl, full.out.weight, full.out.bias, 1, V + 1, 10, exclude=exd)
            v2, i2 = sharded_full_catalogue_topk(hl, full.out.weight, full.out.bias, V, 10, exclude=exd)
            assert torch.equal(i1, i2) and torch.equal(v1, v2)
        q.put((rank, "ok"))
    except Exception:  # noqa
        import traceback
        q.put((rank, traceback.format_exc()))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.timeout(300)
def test_two_gpu_sharded_topk_excluding():
    """A ``shard_bert_model`` model's ``full_catalogue_topk(..., exclude)`` equals the unsharded model's on the same users (ids
    exactly, scores to 1e-6 as in the unfiltered two-GPU test), and ``sharded_full_catalogue_topk(..., exclude)`` equals one call."""
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=280) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    for r in res:
        print("rank", r[0], r[1])
    assert all(r[1] == "ok" for r in res), res
