#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on B200: training sequences/s (BERT4Rec, SASRec) and full-catalogue top-10
evaluation users/s, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload bert|sasrec|eval] [--impl reference] [--dump-outputs DIR]

Workloads (SURVEY.md 8d):
  bert    (default, the headline line) BASELINE configs[1]: BERT4Rec nb=2 d=64 h=2 L=200 mask_prob=0.15, ML-1M-shaped
          synthetic data, B=1024 per GPU; N GPUs = data parallel, weak scaling.
  sasrec  BASELINE configs[2] shape: SASRec nb=2 d=128 h=2 L=50, Amazon-Beauty-shaped synthetic data, B=4096 per GPU.
  eval    BASELINE configs[4] shape: full-catalogue top-10 HR/NDCG over a 10M-item table (SASRec d=64 L=50 nb=2),
          16384 users per step; N GPUs = item table row-sharded, vocab-parallel top-k merge (strong scaling).
A "step" is one full optimisation step (zero_grad, forward, fused loss, backward, dense Adam) over one batch, or one
evaluation batch (transformer body, fused scoring + top-10, HR/NDCG).  One JSON line is printed by rank 0:
  value        whole-job units/s with the inputs already resident in HBM (CUDA-event timed, max over ranks)
  e2e          the same through the public trainer / model API from pinned HOST buffers (H2D of the batch and the D2H
               read of the loss / metric values inside the timed region, every step)
  roofline     the dominant entry point of the step: algorithmic FLOP (or bytes) / its measured launch time vs the
               measured peak in MEASURED_PEAKS.json
  cpu_baseline the reference's own classes (baseline/_ref, kind "reference"; oracle port otherwise) timed on this box's
               host cores on a bounded sample of the same workload
  extra        (default workload) the other two workloads as full sub-lines, and the north-star multi-GPU layouts at
               THIS world size: sharded 10M-item evaluation, SASRec cfg3 strong scaling (global B=4096), BERT4Rec
               configs[3] (d=256, 1M items) with row-sharded tables -- each with a single-GPU-equivalence check.
`--impl reference` times only the CPU arm (rank 0) and prints the same line with "impl": "reference".
`--dump-outputs DIR` writes what the top-level workload's last timed step returned, as DIR/<name>.npy (rank 0): for training
the loss plus every parameter and gradient after that step, for evaluation the top-10 values / ids and the metric means.
The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SPECS = {
    "bert": dict(name="BERT4Rec nb=2 d=64 h=2 L=200 mask_prob=0.15 V=3416 (BASELINE configs[1], ML-1M-shaped synthetic)", kind="bert",
                 num_users=6040, V=3416, mean_len=165, min_len=20, L=200, d=64, nb=2, h=2, mask_prob=0.15, dropout=0.1, batch=1024,
                 cpu_batch=64, metric="train_sequences_per_s", unit="seq/s"),
    "sasrec": dict(name="SASRec nb=2 d=128 h=2 L=50 V=12101, 1 sampled negative per position (BASELINE configs[2] shape, Amazon-Beauty-shaped synthetic)",
                   kind="sas", num_users=22363, V=12101, mean_len=8.9, min_len=5, L=50, d=128, nb=2, h=2, dropout=0.2, batch=4096,
                   cpu_batch=128, metric="train_sequences_per_s", unit="seq/s"),
    "eval": dict(name="full-catalogue top-10 HR/NDCG, SASRec nb=2 d=64 h=1 L=50 over a 10,000,000-item table, 16384 users per step "
                      "(BASELINE configs[4] shape)", kind="sas", V=10_000_000, L=50, d=64, nb=2, h=1, users_per_step=16384,
                 metric="eval_users_per_s", unit="users/s"),
}
CFG4 = dict(V=1_000_000, L=200, d=256, nb=4, h=4, dropout=0.1, batch_per_gpu=512)
N_ROT = 4  # distinct batches rotated through the timed region


# ------------------------------------------------------------------------------------------------ helpers
def model_args(spec, device, dropout, batch=None, V=None):
    V = spec["V"] if V is None else V
    common = dict(num_items=V, max_len=spec["L"], device=device, optimizer="Adam", lr=1e-3, weight_decay=0, momentum=None, decay_step=25,
                  gamma=1.0, num_epochs=1, metric_ks=[1, 5, 10], best_metric="NDCG@10", train_batch_size=batch or spec.get("batch", 1),
                  resume_path=None)
    if spec["kind"] == "bert":
        return SimpleNamespace(model_code="bert", model_init_seed=0, bert_num_blocks=spec["nb"], bert_num_heads=spec["h"],
                               bert_hidden_units=spec["d"], bert_dropout=dropout, bert_hidden_dropout=dropout, **common)
    return SimpleNamespace(model_code="sas", sas_hidden_units=spec["d"], sas_num_blocks=spec["nb"], sas_heads=spec["h"], sas_dropout=dropout,
                           l2_emb=0.0, **common)


def make_batches(spec, n_batches, batch, seed):
    """Host batches in the reference's wire format: BERT (tokens, labels) / SASRec (seq, pos, neg), int64 [B, L]."""
    from rbm_b200.dataloaders import synthetic_interactions, sliding_window_partition, BertBatcher, SasBatcher
    hist = synthetic_interactions(spec["num_users"], spec["V"], spec["mean_len"], spec["min_len"], seed=1234)
    ds = sliding_window_partition(hist, spec["L"], 0.3)
    if spec["kind"] == "bert":
        bb = BertBatcher(ds[0], spec["V"], spec["L"], spec["mask_prob"], seed=seed)
    else:
        bb = SasBatcher(ds[0], spec["V"], spec["L"], seed=seed)
    return [tuple(np.ascontiguousarray(x) for x in bb.batch(batch)) for _ in range(n_batches)]


def host_threads():
    # all the host threads this process may use (torchrun exports OMP_NUM_THREADS=1 for its workers: undo that here)
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        n = max(1, os.cpu_count() or 1)
    torch.set_num_threads(n)
    return torch.get_num_threads()


DUMP_LIMIT_BYTES = 64 << 20


def write_outputs(out_dir, arrays):
    """Save {name: tensor} as out_dir/<name>.npy: floating tensors as float32, integer ones (ids) as float64, which holds
    every id below 2^53 exactly."""
    host = {}
    for name, t in arrays.items():
        t = t.detach().cpu()
        host[name] = (t.double() if not t.is_floating_point() else t.float()).numpy()
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# --------------------------------------------------------------------------------------------- CPU reference legs
def cpu_train_leg(spec, steps, warmup):
    """The reference's CPU train step on all host cores: its own model + trainer classes (baseline/_ref) when present,
    the oracle port of the same torch ops otherwise.  -> dict(value, unit, cores, kind, sample, ms)."""
    from baseline import reference_arm as ra
    threads = host_threads()
    B = spec["cpu_batch"]
    batches = make_batches(spec, 2, B, seed=7)
    torch.manual_seed(0)
    if ra.available():
        t = ra.make_trainer(model_args(spec, "cpu", spec["dropout"], batch=B))
        t.model.train()
        if spec["kind"] == "bert":
            feed = [tuple(torch.from_numpy(x) for x in b) for b in batches]
        else:
            feed = batches  # numpy arrays, as WarpSampler yields them (NN/trainers/sas.py:36)
        step = lambda i: ra.train_step(t, feed[i % len(feed)])
        kind, what = "reference", "the reference's own %s + %s.calculate_loss / backward / optim.Adam (baseline/_ref, unmodified)" % (
            "BERTModel" if spec["kind"] == "bert" else "SASModel", "BERTTrainer" if spec["kind"] == "bert" else "SASTrainer")
    else:
        from oracle.common import DropoutPlan
        drop = DropoutPlan(training=True)
        if spec["kind"] == "bert":
            from oracle import bert4rec as om_
            sd = om_.random_state_dict(spec["V"], spec["L"], spec["d"], spec["nb"], seed=0)
        else:
            from oracle import sasrec as om_
            sd = om_.random_state_dict(spec["V"], spec["L"], spec["d"], spec["nb"], seed=0)
        params = {k: torch.nn.Parameter(v.clone()) for k, v in sd.items()}
        opt = torch.optim.Adam(params.values(), lr=1e-3)
        feed = [tuple(torch.from_numpy(x) for x in b) for b in batches]

        def step(i):
            opt.zero_grad()
            if spec["kind"] == "bert":
                loss = om_.loss(params, *feed[i % 2], spec["nb"], spec["h"], p_attn=spec["dropout"], p_hidden=spec["dropout"], drop=drop)
            else:
                loss = om_.loss(params, *feed[i % 2], spec["nb"], spec["h"], p=spec["dropout"], drop=drop)
            loss.backward()
            opt.step()
            return loss.item()
        kind, what = "port", "oracle port of the reference's torch CPU path (baseline/_ref absent)"
    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
    dt = time.perf_counter() - t0
    return {"value": B * steps / dt, "unit": spec["unit"], "cores": threads, "kind": kind, "ms_per_step": dt / steps * 1e3,
            "sample": "%d steps of B=%d of the same workload, dropout %.2f: %s; %.0f ms/step" % (steps, B, spec["dropout"], what, dt / steps * 1e3)}


def cpu_eval_leg(spec, users=48):
    """Full-catalogue evaluation on the host: the reference's SAS.predict gathers [B, V, d] (NN/models/sas_model/sas.py:110),
    which cannot be allocated at 10M items, so the scoring is the oracle port chunked over the catalogue (same fp32 matmul);
    ranking + HR/NDCG are the reference's own recalls_ndcgs_and_mrr_for_ks (full argsort on the CPU) when baseline/_ref exists."""
    from baseline import reference_arm as ra
    from oracle import sasrec as osr
    threads = host_threads()
    V, L, d, nb, h = spec["V"], spec["L"], spec["d"], spec["nb"], spec["h"]
    g = torch.Generator().manual_seed(5)
    sd = osr.random_state_dict(V, L, d, nb, seed=0, scale=1.0)
    seq = torch.randint(1, V + 1, (users, L), generator=g)
    pos = torch.randint(1, V + 1, (users,), generator=g)
    if ra.available():
        metric_fn, kind = ra.modules()[3], "port+reference"
    else:
        from oracle.metrics import recalls_ndcgs_and_mrr_for_ks as metric_fn
        kind = "port"
    t0 = time.perf_counter()
    with torch.no_grad():
        scores = osr.scores_full_catalogue(sd, seq, nb, h)  # [users, V] (items 1..V), chunked fp32 matmul
        labels = torch.zeros(users, V, dtype=torch.long)
        labels[torch.arange(users), pos - 1] = 1
        metric_fn(scores, labels, [10])
    dt = time.perf_counter() - t0
    return {"value": users / dt, "unit": spec["unit"], "cores": threads, "kind": kind, "ms_per_step": dt * 1e3,
            "sample": "%d users x %d items: chunked fp32 scoring (oracle port of SAS.predict; the reference's [B,V,d] gather cannot be "
                      "allocated at this V) + %s recalls_ndcgs_and_mrr_for_ks (full argsort); %.1f s" % (
                          users, V, "the reference's own" if ra.available() else "the oracle's", dt)}


def run_reference(args, rank):
    if rank != 0:
        return
    spec = SPECS[args.workload]
    if args.workload == "eval":
        cpu = cpu_eval_leg(spec)
        steps, warmup, cfg = 1, 0, {"workload": spec["name"], "users_per_step": 16}
    else:
        steps, warmup = max(1, min(args.steps, 10)), max(1, min(args.warmup, 2))
        cpu = cpu_train_leg(spec, steps, warmup)
        cfg = {"workload": spec["name"], "batch_per_step": spec["cpu_batch"]}
    cfg["note"] = "CPU, bounded sample of the same workload"
    v = cpu["value"]
    line = {"impl": "reference", "metric": spec["metric"], "value": v, "unit": spec["unit"], "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": cpu["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")},
            "e2e": {"value": v, "unit": spec["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.proc, self.lines = None, []
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ roofline leg
def kernel_work(name, a, shapes):
    """ALGORITHMIC work of one launch of a C-ABI entry point given its call arguments `a` (DESIGN.md 'kernels'):
    ('tensor', FLOP) for the contraction kernels, ('hbm', bytes) for the streaming ones, None if not modelled."""
    if name in ("rbm_attn_fwd", "rbm_attn_bwd"):
        o = 10 if name == "rbm_attn_fwd" else 18
        B, Ln, h, dk, mode = a[o:o + 5]
        pairs = Ln * (Ln + 1) / 2 if mode == 1 else Ln * Ln  # causal touches half the score matrix
        return "tensor", (4.0 if name == "rbm_attn_fwd" else 10.0) * pairs * dk * B * h
    if name in ("rbm_attn_fwd_lq", "rbm_attn_bwd_lq"):  # Lq compacted queries per sequence against all L keys
        o = 10 if name == "rbm_attn_fwd_lq" else 18
        B, Ln, Lq, h, dk = a[o:o + 5]
        return "tensor", (4.0 if name == "rbm_attn_fwd_lq" else 10.0) * Lq * Ln * dk * B * h
    if name == "rbm_ce_fwd":
        return "tensor", 2.0 * shapes["P"] * a[9] * a[10]
    if name == "rbm_ce_bwd":
        return "tensor", 4.0 * shapes["P"] * a[12] * a[13]
    if name == "rbm_score_topk":
        return "tensor", 2.0 * a[9] * a[10] * (a[5] - a[4])  # 2 * U * d * items
    # Linear family at d = 64..256: arithmetic intensity of a few FLOP/B -> HBM-bound; algorithmic bytes = every operand
    # and result once (DESIGN.md section 3)
    if name in ("rbm_attn_live_fwd", "rbm_attn_live_bwd"):
        # compact SASRec attention: a (sequence, head) item is ~ len^2 / 2 scores of d_k = 64 -- latency / instruction bound, reported
        # against the bytes it has to move: q, k|v, out (+ dout, dq, dk|dv, the padding-key rows in the backward) of the live rows
        o = 10 if name == "rbm_attn_live_fwd" else 16
        h, dk = a[o + 2], a[o + 3]
        return "hbm", (4.0 if name == "rbm_attn_live_fwd" else 10.0) * shapes.get("live_rows", 0.0) * h * dk * 4
    if name in ("rbm_linear_fwd", "rbm_linear_fwd_ws"):
        M, N, K = a[7], a[8], a[9]
        return "hbm", 4.0 * (M * K + N * K + M * N * (1 + (1 if a[6] else 0) + (1 if a[11] else 0)))  # + pre-activation, + residual
    if name == "rbm_linear_bwd_data":
        M, N, K = a[5], a[6], a[7]
        return "hbm", 4.0 * (M * N + N * K + M * K)
    if name == "rbm_linear_bwd_weight":
        M, N, K = a[6], a[7], a[8]
        return "hbm", 4.0 * (M * N + M * K + N * K)
    if name in ("rbm_layernorm_fwd", "rbm_layernorm_bwd"):
        rows, d = (a[5], a[6]) if name == "rbm_layernorm_fwd" else (a[7], a[8])
        return "hbm", (2.0 if name == "rbm_layernorm_fwd" else 3.0) * rows * d * 4
    if name == "rbm_linear_epilogue_bwd":
        return "hbm", 3.0 * a[4] * a[5] * 4
    if name == "rbm_adam_multi":
        return "hbm", 28.0 * shapes["n_params"]
    if name == "rbm_embed_fwd":
        return "hbm", a[4] * (8.0 + 2 * a[6] * 4)
    return None


def roofline_from_profile(prof, n_steps, shapes, peaks, traffic_key=None):
    """Per-entry-point CUDA-event times of `n_steps` eager steps -> (roofline of the dominant entry point, time shares,
    compact rooflines of the top entry points)."""
    totals = {k: sum(ms for ms, _ in v) / n_steps for k, v in prof.items()}
    step_ms = sum(totals.values())
    top = max(totals, key=totals.get)

    def roof(name):
        works = [kernel_work(name, a, shapes) for _, a in prof[name]]
        if not works or any(w is None for w in works):
            return None
        kind = works[0][0]
        amount = sum(w[1] for w in works)
        tot_ms = sum(ms for ms, _ in prof[name])
        if kind == "tensor":
            peak, unit, ach = peaks.get("bf16_tflops_sustained", 1400.0), "TFLOP/s", amount / (tot_ms * 1e-3) / 1e12
            src = "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback 1.4 PFLOP/s sustained"
        else:
            peak, unit, ach = peaks.get("hbm_gbs", 6650.0), "GB/s", amount / (tot_ms * 1e-3) / 1e9
            src = "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s"
        return {"kernel": name, "bound": kind, "achieved": ach, "peak": peak, "unit": unit, "frac": ach / peak, "traffic": None,
                "peak_source": src, "launches_per_step": len(works) / n_steps, "avg_launch_ms": tot_ms / len(works),
                "share_of_step": totals[name] / step_ms}

    r = roof(top)
    if r is not None:
        for fn in ("r2_traffic.json", "r1_traffic.json"):  # DRAM bytes per launch from the committed `ncu --set full` captures
            try:
                t = json.load(open(os.path.join(ROOT, "profiles", fn))).get(traffic_key or top)
                if t is not None:
                    r["traffic"] = t["bytes"] if isinstance(t, dict) else t
                    break
            except Exception:
                pass
        if r["bound"] == "tensor":
            r["note"] = ("fp32-parity arithmetic (split-precision passes on the tensor cores); algorithmic FLOP over the bf16 tensor-pipe "
                         "peak on purpose")
    shares = {k: round(v / step_ms, 4) for k, v in sorted(totals.items(), key=lambda kv: -kv[1])[:8]}
    compact = {}
    for k in sorted(totals, key=totals.get, reverse=True)[:8]:
        rr = roof(k)
        compact[k] = None if rr is None else {"bound": rr["bound"], "achieved": round(rr["achieved"], 3), "unit": rr["unit"], "frac": round(rr["frac"], 5)}
    return r, shares, compact


class Ctx:
    """Rank / device / timing helpers shared by the workloads."""

    def __init__(self, args):
        import torch.distributed as dist
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU leg"
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = dist
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        self.peaks = load_peaks()

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps):
        """ms for `steps` calls: barrier + synchronize on both sides, CUDA events, max over ranks."""
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return ms.item()

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


# ------------------------------------------------------------------------------------- training workloads (bert / sasrec)
def train_workload(ctx, key, steps, warmup, batch=None, with_cpu=True, with_roofline=True, global_batch=None, check_equivalence=False,
                   dump=None):
    """One training line.  Data parallel over ctx.world ranks: weak scaling with `batch` sequences per GPU, or strong
    scaling when `global_batch` is given (each rank takes global_batch / world sequences).  `dump`: directory that gets
    the loss, parameters and gradients of the last timed step (rank 0)."""
    import rbm_b200
    from rbm_b200 import lib as L
    from rbm_b200.dist import GradSync, decorrelate_dropout
    args, world, rank, dev = ctx.args, ctx.world, ctx.rank, ctx.dev
    spec = SPECS[key]
    Bsz = (global_batch // world) if global_batch else (batch or spec["batch"])
    margs = model_args(spec, str(dev), spec["dropout"], batch=Bsz)
    torch.manual_seed(1234)  # SASRec does not seed itself (SURVEY 8a a1): identical replicas need the same torch seed
    model = rbm_b200.model_factory(margs)
    trainer = rbm_b200.trainer_factory(margs, model, None, None, None, None)
    model.train()
    equiv = None
    if check_equivalence and world > 1:
        equiv = dp_equivalence(ctx, spec, Bsz)
    if world > 1:
        decorrelate_dropout(model)  # every rank its own dropout stream (the ranks are built from the same seeds)
        if not os.environ.get("RBM_BENCH_NO_GRADSYNC"):  # diagnostic: N independent replicas (per-rank speed without the exchange)
            trainer.dist_sync = GradSync(model.parameters())
    raw = make_batches(spec, N_ROT, Bsz, seed=100 + rank)
    host = [tuple(torch.from_numpy(x).pin_memory() for x in b) for b in raw]
    devb = [tuple(x.to(dev) for x in b) for b in host]

    last = {}

    def step_dev(i):
        # detached: a loss that kept its autograd graph alive into capture_train_step would invalidate the capture
        last["loss"] = trainer.train_step(devb[i % N_ROT]).detach()

    step_mode = args.step_mode
    if step_mode == "graph":
        for i in range(2):
            step_dev(i)  # eager first: one-time lazy work and the NCCL communicator
        try:
            trainer.capture_train_step(devb[0], collective=args.dp_collective)
        except Exception as ex:  # all ranks fail alike (same code path); the eager step is the same arithmetic
            if rank == 0:
                print("capture_train_step failed (%r): eager steps" % (ex,), file=sys.stderr)
            step_mode = "eager"
    for i in range(warmup):
        step_dev(i)
    L.launch_count = 0
    sampler = ClockSampler(ctx.local_rank) if rank == 0 else None
    ms_dev = ctx.timed(step_dev, steps)
    launches = L.launch_count
    clocks = sampler.stop() if sampler else None
    if dump and rank == 0:
        outs = {"loss": last["loss"]}
        for k, p in model.named_parameters():
            outs["param." + k] = p
            if p.grad is not None:
                outs["grad." + k] = p.grad
        write_outputs(dump, outs)

    # ---- end-to-end leg: host pinned buffers -> trainer API -> loss value back on the host, every step
    losses = []

    def step_e2e(i):
        losses.append(trainer.train_step(host[i % N_ROT]).item())

    for i in range(3):
        step_e2e(i)
    ms_e2e = ctx.timed(step_e2e, steps)
    h2d = sum(x.numel() * x.element_size() for x in host[0])
    trainer.release_train_graph()
    if rank != 0:
        return None
    trainer.dist_sync = None  # the other ranks are done: no collectives from here on

    roofline = shares = compact = None
    if with_roofline:
        # per-entry-point CUDA-event timing of a few eager steps (rank 0)
        L.profile = {}
        for i in range(3):
            step_dev(i)
        prof = L.profile_collect()
        L.profile = None
        shapes = dict(B=Bsz, L=spec["L"], d=spec["d"], h=spec["h"], nb=spec["nb"], V1=spec["V"] + 1,
                      n_params=sum(p.numel() for p in model.parameters()))
        if spec["kind"] == "bert":
            shapes["P"] = float(np.mean([(b[1] != 0).sum() for b in raw]))
        else:
            shapes["live_rows"] = float(np.mean([(b[0] != 0).sum() for b in raw]))
        roofline, shares, compact = roofline_from_profile(prof, 3, shapes, ctx.peaks)

    cpu = None
    if with_cpu and world == 1 and not args.no_cpu_baseline:
        c = cpu_train_leg(spec, steps=6, warmup=1)
        cpu = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")}

    total = Bsz * world * steps
    line = {"metric": spec["metric"], "value": total / (ms_dev * 1e-3), "unit": spec["unit"], "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "strong" if global_batch else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": spec["name"], "batch_per_gpu": Bsz, "global_batch": Bsz * world, "seq_len": spec["L"],
                       "dropout": spec["dropout"], "optimizer": "Adam (dense, fused)", "parallelism": "dp%d" % world,
                       "step": ("one CUDA graph per step (trainer.capture_train_step)" if world == 1 else
                                "two CUDA graphs + one eager NCCL all-reduce of the flat gradient bucket per step" if args.dp_collective == "split"
                                else "one CUDA graph per step incl. the NCCL all-reduce") if step_mode == "graph" else "eager launches",
                       "l2_policy": "per-step working set (activations + saved tensors, GBs) exceeds the 126 MB L2; %d distinct batches rotate" % N_ROT},
            "e2e": {"value": total / (ms_e2e * 1e-3), "unit": spec["unit"], "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": ms_e2e / steps},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "kernel_time_shares": shares,
            "roofline_by_entry_point": compact, "cpu_baseline": cpu, "final_loss": losses[-1] if losses else None}
    if spec["kind"] == "bert":
        line["config"]["label_rows"] = ("%.1f %% of the positions are labelled; the final block's attention queries, output projection, "
                                        "LayerNorm, feed-forward and the scoring run on those rows only (exact: the loss reads no other "
                                        "row of that block)" % (100 * float(np.mean([(b[1] != 0).mean() for b in raw]))))
    if spec["kind"] == "sas":
        frac = float(np.mean([(b[0] != 0).mean() for b in raw]))
        cap = getattr(trainer, "_graph_row_cap", 0) if step_mode == "graph" else None
        line["config"]["live_rows"] = ("%.1f %% of the positions are non-padding; LayerNorm / Linear / feed-forward / attention / embedding "
                                       "gradient run on those rows only (exact: the reference multiplies padding rows by zero after every "
                                       "block; captured row capacity %s of %d)" % (100 * frac, cap, Bsz * spec["L"]))
    if equiv is not None:
        line["single_gpu_equivalence"] = equiv
    del trainer, model
    torch.cuda.empty_cache()
    return line


def dp_equivalence(ctx, spec, Bsz):
    """N ranks == 1 rank on the same global batch (SURVEY 8e), dropout off: the count-weighted mean of the ranks' losses on
    their slices against rank 0's loss on the concatenated batch (relative difference; the gradient identity is the 2-GPU
    test's job, tests/test_dist_gpu.py)."""
    import rbm_b200
    dist, dev, world, rank = ctx.dist, ctx.dev, ctx.world, ctx.rank
    torch.manual_seed(1234)
    m = rbm_b200.model_factory(model_args(spec, str(dev), 0.0, batch=Bsz)).to(dev).train()
    glob = make_batches(spec, 1, Bsz * world, seed=999)[0]
    sl = slice(rank * Bsz, (rank + 1) * Bsz)
    with torch.no_grad():
        mine = m.loss(*[torch.from_numpy(x[sl]).to(dev) for x in glob])
        cnt = torch.tensor([float((glob[1][sl] != 0).sum())], device=dev)
        acc = torch.cat([mine.reshape(1) * cnt, cnt])
        dist.all_reduce(acc)
        out = None
        if rank == 0:
            full = m.loss(*[torch.from_numpy(x).to(dev) for x in glob]).item()
            got = float(acc[0] / acc[1])
            out = {"loss_n_ranks": got, "loss_one_rank": full, "rel_diff": abs(got - full) / abs(full), "ok": abs(got - full) <= 1e-5 * abs(full)}
    del m
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------- evaluation workload
def eval_workload(ctx, steps, warmup, with_cpu=True, V=None, dump=None):
    """Full-catalogue top-10 HR/NDCG users/s.  world == 1: the whole item table on one GPU.  world > 1: the table is
    row-sharded (shard_sas_model), every rank brings users_per_step / world users per step; last hidden rows all-gathered,
    shard-local fused scoring + top-10 with global ids, all-to-all of the lists by user range, merge, HR/NDCG partial sums
    all-reduced.  Check: ids of rank 0's first users equal to the unsharded model's (computed before the table is cut)."""
    import rbm_b200
    from rbm_b200 import lib as L, ops
    from rbm_b200.dist import shard_sas_model
    from rbm_b200.trainers.utils import _as_dict
    args, world, rank, dev, dist = ctx.args, ctx.world, ctx.rank, ctx.dev, ctx.dist
    spec = SPECS["eval"]
    V = spec["V"] if V is None else V
    U, Ln, d = spec["users_per_step"], spec["L"], spec["d"]
    Ul = U // world
    torch.manual_seed(4321)  # identical tables on every rank before the cut
    with torch.device(dev):
        model = rbm_b200.model_factory(model_args(spec, str(dev), 0.0, V=V))
    model = model.to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(77)
    seq_glob = [torch.randint(1, V + 1, (U, Ln), device=dev, generator=g) for _ in range(2)]
    pos_glob = [torch.randint(1, V + 1, (U,), device=dev, generator=g) for _ in range(2)]
    equiv = None
    if world > 1:
        n_chk = min(256, Ul)
        ref_ids = None
        if rank == 0:
            with torch.no_grad():
                _, ref_ids = model.full_catalogue_topk(seq_glob[0][:n_chk], 10)
        shard_sas_model(model)
        torch.cuda.empty_cache()
    sl = slice(rank * Ul, (rank + 1) * Ul)
    seqs = [s[sl].contiguous() for s in seq_glob]
    poss = [p[sl].contiguous() for p in pos_glob]
    host = [(s.cpu().pin_memory(), p.cpu().pin_memory()) for s, p in zip(seqs, poss)]

    def metrics_dev(ids, positives):
        per_user = ops.rank_metrics(ids, [10], positives=positives)
        means = ops.column_mean(per_user)  # [3] = Recall@10, NDCG@10, MRR@10 of this rank's users
        if world > 1:
            dist.all_reduce(means)
            means = means / world
        return means

    last_dev = {}

    def step_dev(i):
        with torch.no_grad():
            vals, ids = model.full_catalogue_topk(seqs[i % 2], 10)
            last_dev.update(top10_values=vals, top10_ids=ids, metric_means=metrics_dev(ids, poss[i % 2]))

    if world > 1:
        with torch.no_grad():
            _, ids0 = model.full_catalogue_topk(seqs[0], 10)
        if rank == 0:
            same = bool(torch.equal(ids0[:n_chk], ref_ids))
            equiv = {"users_checked": n_chk, "top10_ids_equal_to_unsharded": same, "ok": same}
    for i in range(max(1, warmup)):
        step_dev(i)
    L.launch_count = 0
    sampler = ClockSampler(ctx.local_rank) if rank == 0 else None
    ms_dev = ctx.timed(step_dev, steps)
    launches = L.launch_count
    clocks = sampler.stop() if sampler else None
    if dump and rank == 0:
        write_outputs(dump, last_dev)
    last = {}

    def step_e2e(i):
        s, p = host[i % 2]
        with torch.no_grad():
            _, ids = model.full_catalogue_topk(s.to(dev, non_blocking=True), 10)
            last["m"] = _as_dict([10], metrics_dev(ids, p.to(dev, non_blocking=True)).tolist())

    step_e2e(0)
    ms_e2e = ctx.timed(step_e2e, steps)
    if rank != 0:
        return None
    # roofline: the fused scoring + top-k entry point (per-call CUDA events, rank 0; collectives are not entered again)
    roofline = None
    if world == 1:
        L.profile = {}
        for i in range(2):
            step_dev(i)
        prof = L.profile_collect()
        L.profile = None
        roofline, shares, _ = roofline_from_profile(prof, 2, {}, ctx.peaks, traffic_key="rbm_score_topk_10M")
        if roofline is not None and roofline.get("kernel") == "rbm_score_topk":
            # every one of the U x V scores leaves tensor memory through tcgen05.ld: 16 B/clk per SM sub-partition (B300_MICROARCH.md
            # "TMEM-read 64 B/cyc" per SM; reproduced here: 2069 cycles per 256-user x 128-item tile against 2048 for its 128 KB)
            sm_hz = (clocks or {}).get("sm_mhz") or 1965.0
            tmem_floor_ms = U * V / world * 4.0 / (148 * 64.0 * sm_hz * 1e6) * 1e3
            roofline["note"] = ("single-pass fp16 selection (kind::f16) + exact fp32 re-score; algorithmic 2*d*V FLOP per user over the bf16 "
                                "tensor-pipe peak.  The binding resource is the tensor-memory read path: every score is read once at 64 B/clk/SM")
            roofline["tmem_read_bound"] = {"floor_ms_per_step": tmem_floor_ms, "frac": tmem_floor_ms / roofline["avg_launch_ms"],
                                           "model": "U*V*4 B / (148 SMs x 64 B/clk x SM clock)"}
    cpu = None
    if with_cpu and world == 1 and not args.no_cpu_baseline:
        c = cpu_eval_leg(dict(spec, V=V))
        cpu = {k: c[k] for k in ("value", "unit", "cores", "kind", "sample")}
    line = {"metric": spec["metric"], "value": U * steps / (ms_dev * 1e-3), "unit": spec["unit"], "n_gpus": world, "steps": steps,
            "warmup": max(1, warmup), "ms_per_step": ms_dev / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": spec["name"] if V == spec["V"] else spec["name"].replace("10,000,000", "{:,}".format(V)),
                       "users_per_step": U, "users_per_gpu": Ul, "items": V, "k": 10,
                       "parallelism": "1 GPU, whole table" if world == 1 else "item table row-sharded over %d GPUs (vocab-parallel top-k merge), users data-parallel" % world,
                       "arithmetic": "single-pass fp16 candidate selection (range-scaled copies) with a per-user error certificate, exact fp32 re-score / re-scan: ids equal the fp32 ranking",
                       "l2_policy": "the item-table shard (%.2f GB) exceeds the 126 MB L2" % (V * d * 4 / world / 1e9)},
            "e2e": {"value": U * steps / (ms_e2e * 1e-3), "unit": spec["unit"], "h2d_bytes_per_step": Ul * Ln * 8 + Ul * 8,
                    "d2h_bytes_per_step": 12, "ms_per_step": ms_e2e / steps},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
            "logits_per_s": U * V * steps / (ms_dev * 1e-3), "metrics_last_step": last.get("m")}
    if equiv is not None:
        line["single_gpu_equivalence"] = equiv
    del model
    torch.cuda.empty_cache()
    return line


# ------------------------------------------------------------ BERT4Rec configs[3]: d=256, 1M items, row-sharded tables
def cfg4_workload(ctx, steps=5):
    """BASELINE configs[3]: BERT4Rec nb=4 d=256 h=4 L=200, full softmax over 1M items; token table and output layer
    row-sharded over the ranks (shard_bert_model), body data-parallel, CFG4['batch_per_gpu'] sequences per GPU (weak).
    Check (eval mode, no dropout): the sharded loss of the global batch against rank 0's unsharded model."""
    import rbm_b200
    from rbm_b200.dist import GradSync, shard_bert_model, replicated_parameters
    world, rank, dev, dist = ctx.world, ctx.rank, ctx.dev, ctx.dist
    c = CFG4
    V, Ln, Bl = c["V"], c["L"], c["batch_per_gpu"]
    spec = dict(kind="bert", V=V, L=Ln, d=c["d"], nb=c["nb"], h=c["h"])
    margs = model_args(spec, str(dev), c["dropout"], batch=Bl)
    with torch.device(dev):
        model = rbm_b200.model_factory(margs)
    model = model.to(dev)
    g = torch.Generator(device=dev).manual_seed(4)
    glob = []
    for _ in range(2):
        tok = torch.randint(1, V + 1, (Bl * world, Ln), device=dev, generator=g)
        lab = torch.where(torch.rand(Bl * world, Ln, device=dev, generator=g) < 0.15, tok, torch.zeros_like(tok))
        glob.append((torch.where(lab != 0, torch.full_like(tok, V + 1), tok), lab))
    sl = slice(rank * Bl, (rank + 1) * Bl)
    equiv = None
    ref_loss = None
    if world > 1:
        # equivalence on a small global batch (32 sequences per rank), eval mode (no dropout): unsharded (rank 0, before the
        # tables are cut) vs sharded
        nb_chk = 32
        chk = tuple(x[:nb_chk * world] for x in glob[0])
        model.eval()
        if rank == 0:
            with torch.no_grad():
                ref_loss = model.loss(*chk).item()
    shard_bert_model(model, capacity=int(0.25 * Bl * Ln))
    torch.cuda.empty_cache()
    if world > 1:
        with torch.no_grad():
            got = model.loss(*(x[rank * nb_chk:(rank + 1) * nb_chk] for x in chk)).item()
        if rank == 0:
            equiv = {"loss_sharded": got, "loss_unsharded": ref_loss, "rel_diff": abs(got - ref_loss) / abs(ref_loss),
                     "ok": abs(got - ref_loss) <= 1e-5 * abs(ref_loss), "sequences_checked": nb_chk * world}
    model.train()
    trainer = rbm_b200.trainer_factory(margs, model, None, None, None, None)
    if world > 1:
        trainer.dist_sync = GradSync(replicated_parameters(model))
    batches = [tuple(x[sl].contiguous() for x in b) for b in glob]
    del glob
    t0 = time.perf_counter()
    trainer.train_step(batches[0])
    torch.cuda.synchronize()
    first_s = time.perf_counter() - t0
    if first_s > 8.0:  # a step this slow means the d=256 scoring kernels are not on the tensor path: report it and stop
        ms = first_s * 1e3
        steps_done = 1
    else:
        trainer.train_step(batches[1])
        ms = ctx.timed(lambda i: trainer.train_step(batches[i % 2]), steps) / steps
        steps_done = steps
    # optional reduced-precision line (clearly labelled; the headline stays fp32-parity): the scoring + cross-entropy kernels with
    # ONE fp16 pass per product instead of three (RBM_CE_WIDE_PASSES=1; 1e-3 parity test: tests/test_kernels_gpu.py
    # test_score_ce_wide_million_items[1])
    ms_fast = None
    if steps_done > 1:
        os.environ["RBM_CE_WIDE_PASSES"] = "1"
        try:
            trainer.train_step(batches[0])
            ms_fast = ctx.timed(lambda i: trainer.train_step(batches[i % 2]), steps) / steps
        finally:
            os.environ.pop("RBM_CE_WIDE_PASSES", None)
    trainer._check_shard_overflow()
    out = None
    if rank == 0:
        P = 0.15 * Bl * world * Ln
        flop = 6.0 * c["d"] * (V + 1) * P / world + 3.0 * c["nb"] * (24 * Ln * c["d"] ** 2 + 4 * Ln * Ln * c["d"]) * Bl
        out = {"config": "BERT4Rec nb=4 d=256 h=4 L=200 V=1,000,000, dropout 0.1, %d sequences per GPU (global batch %d), token table + output layer "
                         "row-sharded over %d GPU(s), body data-parallel, dense Adam on the shards (BASELINE configs[3])" % (Bl, Bl * world, world),
               "seq_per_s": Bl * world / (ms * 1e-3), "ms_per_step": ms, "timed_steps": steps_done, "scaling": "weak",
               "algorithmic_tflops_per_gpu": flop / (ms * 1e-3) / 1e12,
               "frac_of_bf16_peak": flop / (ms * 1e-3) / 1e12 / ctx.peaks.get("bf16_tflops_sustained", 1400.0),
               "single_gpu_equivalence": equiv,
               "reduced_precision_line": None if ms_fast is None else {
                   "dtype": "f16 single pass in the scoring + cross-entropy products (fp32 accumulate); everything else as the headline",
                   "seq_per_s": Bl * world / (ms_fast * 1e-3), "ms_per_step": ms_fast,
                   "parity": "loss 1e-4, gradients 1e-3 of scale vs fp64 (test_score_ce_wide_million_items[1])"}}
    del trainer, model
    torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------ small single-GPU extras
def small_extras(dev):
    """B = 128 (the reference's batch size) eager vs CUDA graph, and device-side batch construction (SURVEY 8(f) #1)."""
    import rbm_b200
    from rbm_b200 import ops as ops_mod
    from rbm_b200.dataloaders import synthetic_interactions, sliding_window_partition, DeviceBertTrainLoader, BertBatcher
    out = {}
    spec = SPECS["bert"]

    def ev_time(fn, n):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            fn(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    try:
        Bs = 128
        ma = model_args(spec, str(dev), spec["dropout"], batch=Bs)
        mdl = rbm_b200.model_factory(ma)
        trn = rbm_b200.trainer_factory(ma, mdl, None, None, None, None)
        mdl.train()
        bs = [tuple(torch.from_numpy(x).to(dev) for x in b) for b in make_batches(spec, 4, Bs, seed=55)]
        for i in range(5):
            trn.train_step(bs[i % 4])
        ms_eager = ev_time(lambda i: trn.train_step(bs[i % 4]), 30)
        trn.capture_train_step(bs[0])
        for i in range(3):
            trn.train_step(bs[i % 4])
        ms_graph = ev_time(lambda i: trn.train_step(bs[i % 4]), 30)
        trn.release_train_graph()
        out["small_batch_cuda_graph"] = {"config": "BERT4Rec cfg2 model, B=%d (the reference's default batch size), full optimisation step" % Bs,
                                         "eager_seq_per_s": Bs / ms_eager * 1e3, "eager_ms_per_step": ms_eager,
                                         "graph_seq_per_s": Bs / ms_graph * 1e3, "graph_ms_per_step": ms_graph}
        del trn, mdl
    except Exception as ex:
        out["small_batch_cuda_graph"] = {"error": repr(ex)}
    try:
        Vb, Lb, Bb = spec["V"], spec["L"], spec["batch"]
        hist = synthetic_interactions(6040, Vb, 165.0, 20, seed=1234)
        ds = sliding_window_partition(hist, Lb, 0.3)
        loader = DeviceBertTrainLoader(ds[0], Lb, spec["mask_prob"], Vb, Bb, dev, seed=1)
        users = torch.randint(0, loader.num_users, (Bb,), device=dev)
        dev_batch = lambda i: ops_mod.bert_cloze_batch(loader.ptr, loader.items, users, Lb, spec["mask_prob"], Vb + 1, Vb, 1, i)
        for i in range(3):
            dev_batch(i)
        ms_dev_b = ev_time(dev_batch, 50)
        hb = BertBatcher(ds[0], Vb, Lb, spec["mask_prob"], seed=1)
        t0 = time.perf_counter()
        for _ in range(3):
            hb.batch(Bb)
        ms_host_b = (time.perf_counter() - t0) * 1000 / 3
        out["batch_construction"] = {"config": "BERT4Rec Cloze batch B=%d L=%d from a CSR of %d user windows" % (Bb, Lb, loader.num_users),
                                     "device_ms_per_batch": ms_dev_b, "device_batches_per_s": 1000.0 / ms_dev_b,
                                     "host_numpy_ms_per_batch": ms_host_b, "bytes_per_batch": 2 * Bb * Lb * 8}
    except Exception as ex:
        out["batch_construction"] = {"error": repr(ex)}
    torch.cuda.empty_cache()
    return out


def guarded(ctx, name, fn):
    """Run a secondary measurement; a failure must never break the headline line.  Under N > 1 every rank runs the same code,
    so an exception that is a function of the code path (not of the rank) is raised on all ranks alike."""
    try:
        return fn()
    except Exception as ex:  # noqa
        import traceback
        traceback.print_exc()
        return {"error": "%s: %r" % (name, ex)}


WATCHDOG = {"done": False}


def start_watchdog(rank, line, extras):
    """The secondary measurements run collectives on every rank; should one of them hang (a rank-specific failure leaves the
    others waiting), the headline line -- already measured -- must still be printed: after the limit rank 0 prints it with the
    extras finished so far and every rank leaves."""
    import threading
    limit = float(os.environ.get("RBM_BENCH_EXTRAS_TIMEOUT", "480"))

    def fire():
        if WATCHDOG["done"]:
            return
        if rank == 0:
            done = {k: v for k, v in list(extras.items())}
            done["timeout"] = "secondary measurements exceeded %.0f s; the remaining ones were abandoned" % limit
            line["extra"] = done
            print(json.dumps(line, default=str))
            sys.stdout.flush()
        os._exit(0)

    t = threading.Timer(limit + (0 if rank == 0 else 5), fire)
    t.daemon = True
    t.start()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="bert", choices=sorted(SPECS))
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--step-mode", default=os.environ.get("RBM_BENCH_STEP_MODE", "graph"), choices=["graph", "eager"],
                    help="graph: trainer.capture_train_step (CUDA-graph replay of the whole optimisation step); eager: launch by launch")
    ap.add_argument("--dp-collective", default=os.environ.get("RBM_BENCH_DP_COLLECTIVE", "split"), choices=["split", "graph"],
                    help="N>1 with --step-mode graph: eager NCCL all-reduce between two graphs (split) or captured inside one graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of the top-level workload to DIR/<name>.npy")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        return run_reference(args, rank)
    if args.warmup < 3:
        args.warmup = 3
    ctx = Ctx(args)
    world = ctx.world

    if args.workload == "eval":
        line = eval_workload(ctx, steps=args.steps, warmup=min(args.warmup, 3), dump=args.dump_outputs)
    else:
        line = train_workload(ctx, args.workload, args.steps, args.warmup, batch=args.batch, dump=args.dump_outputs)

    extras = None
    if not args.no_extras and args.workload == "bert":
        extras = {}
        start_watchdog(rank, line, extras)
        ev_steps = 5
        if world == 1:
            # the other two quantities BASELINE.json's metric names, as full lines of their own
            extras["sasrec_train"] = guarded(ctx, "sasrec", lambda: train_workload(ctx, "sasrec", 30, 5))
            extras["eval_10M_items"] = guarded(ctx, "eval", lambda: eval_workload(ctx, steps=ev_steps, warmup=2))
            extras.update(small_extras(ctx.dev))
        else:
            extras["eval_10M_items_sharded"] = guarded(ctx, "eval", lambda: eval_workload(ctx, steps=ev_steps, warmup=2, with_cpu=False))
        # north-star multi-GPU layouts at this world size (the N=1 run provides the first point of each curve)
        extras["sasrec_cfg3_strong_scaling_B4096"] = guarded(ctx, "cfg3 strong", lambda: train_workload(
            ctx, "sasrec", 30, 5, with_cpu=False, with_roofline=False, global_batch=4096, check_equivalence=True))
        extras["bert_cfg4_sharded"] = guarded(ctx, "cfg4", lambda: cfg4_workload(ctx))
        if rank == 0:
            def slim(x):  # sub-lines: keep what the curves need
                if isinstance(x, dict) and "metric" in x:
                    keep = ("metric", "value", "unit", "n_gpus", "steps", "ms_per_step", "scaling", "config", "e2e", "roofline", "cpu_baseline",
                            "gpu_launches", "single_gpu_equivalence", "logits_per_s", "kernel_time_shares", "metrics_last_step", "final_loss")
                    return {k: x[k] for k in keep if k in x}
                return x
            extras = {k: slim(v) for k, v in extras.items()}
    if rank == 0:
        line["extra"] = extras
        print(json.dumps(line))
        sys.stdout.flush()
    WATCHDOG["done"] = True
    ctx.close()


if __name__ == "__main__":
    main()
