"""Full-catalogue top-10 with and without each user's seen items left out, at the bench's eval shape (U = 16384 users, V = 10^7
items, d = 64): device time of ``ops.score_topk`` plain and with ``exclude``, the calls alternating after warm-up, CUDA events.

Two exclusion sets: ``history`` = a 50-item input sequence per user (random ids, as a user's history relates to a random table),
and ``adversarial`` = the user's own unfiltered top-32 plus 18 random items, so that the seen items are exactly the ones that
reach the candidate lists' insertion path (the situation of a trained model, which scores what it was just fed very high).
The excluded ids are checked against the fp32 oracle on 128 users.  Prints the card and its power limit with the numbers and
one JSON line.  Usage: python tools/time_topk_exclusion.py [reps]"""
import json
import subprocess
import sys

import torch

sys.path.insert(0, ".")
import rbm_b200  # noqa: F401,E402
from rbm_b200 import ops  # noqa: E402
from oracle import metrics as om  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def check(f, table, ex, ids, vals, n=128, chunk=16):
    """ids and scores of the first n users == the canonical top-10 of the fp32 (sequential FMA) scores of the items left."""
    for u0 in range(0, n, chunk):
        sc = om.scores_fp32_sequential(f[u0:u0 + chunk], table[1:])
        sc.scatter_(1, ex[u0:u0 + chunk] - 1, float("-inf"))
        rv, ri = torch.topk(sc, 11, dim=1)
        assert bool((rv[:, :-1] > rv[:, 1:]).all()), "exact ties in the top-11: pick another seed"
        assert torch.equal(ids[u0:u0 + chunk], ri[:, :10] + 1) and torch.equal(vals[u0:u0 + chunk], rv[:, :10]), "mismatch at users %d.." % u0
        del sc


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    torch.manual_seed(0)
    U, V, d, k, L = 16384, 10_000_000, 64, 10, 50
    dev = "cuda"
    f = torch.randn(U, d, device=dev)
    table = torch.randn(V + 1, d, device=dev)
    _, top32 = ops.score_topk(f, table, None, 1, V + 1, 32)  # exact fp32 scan: each user's unfiltered top-32
    sets = {"history": torch.randint(1, V + 1, (U, L), device=dev),
            "adversarial": torch.cat([top32, torch.randint(1, V + 1, (U, L - 32), device=dev)], 1)}
    for name, ex in sets.items():
        vals, ids = ops.score_topk(f, table, None, 1, V + 1, k, exclude=ex)
        check(f, table, ex, ids, vals)
        assert not bool((ids.unsqueeze(2) == ex.unsqueeze(1)).any())  # no user is offered one of its own excluded items
    calls = {"plain": lambda: ops.score_topk(f, table, None, 1, V + 1, k)}
    for name, ex in sets.items():
        calls[name] = (lambda e: lambda: ops.score_topk(f, table, None, 1, V + 1, k, exclude=e))(ex)
    for c in calls.values():  # warm-up
        c()
    torch.cuda.synchronize()
    times = {n: [] for n in calls}
    for _ in range(reps):
        for n, c in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            c()
            e1.record()
            e1.synchronize()
            times[n].append(e0.elapsed_time(e1))
    med = {n: sorted(t)[len(t) // 2] for n, t in times.items()}
    gpu = card()
    print("card: %s" % gpu)
    for n in calls:
        print("%-12s median %.2f ms  min %.2f  max %.2f  (%+.1f %% vs plain)" % (n, med[n], min(times[n]), max(times[n]),
                                                                              100.0 * (med[n] / med["plain"] - 1.0)))
    print(json.dumps({"card": gpu, "U": U, "V": V, "d": d, "k": k, "n_excl": L, "reps": reps, "median_ms": med,
                      "oracle_users_checked": 128}))


if __name__ == "__main__":
    main()
