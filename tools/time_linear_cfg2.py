"""Per-entry-point device times of the four Linear layers of a BERT4Rec configs[1] block (M = 1024 x 200 rows, d = 64), forward and
backward, with the epilogues the model uses.  Used to compare kernel choices: run it on each build and compare."""
import sys
import torch
sys.path.insert(0, ".")
import rbm_b200  # noqa: F401
from rbm_b200 import ops, lib as L
torch.manual_seed(0)
M = int(sys.argv[1]) if len(sys.argv) > 1 else 204800
d = int(sys.argv[2]) if len(sys.argv) > 2 else 64
dev = "cuda"
layers = [("qkv", 3 * d, d, dict()), ("out-proj", d, d, dict(pA=0.1, siteA=1, res=True)),
          ("ffn-1", 4 * d, d, dict(act=L.ACT_GELU_TANH, pA=0.1, siteA=2)), ("ffn-2", d, 4 * d, dict(pA=0.1, siteA=3, pB=0.1, siteB=4, res=True))]
for name, N, K, kw in layers:
    x = torch.randn(M, K, device=dev, requires_grad=True)
    w = (torch.randn(N, K, device=dev) * 0.1).requires_grad_(True)
    b = torch.randn(N, device=dev, requires_grad=True)
    res = torch.randn(M, N, device=dev, requires_grad=True) if kw.get("res") else None
    dy = torch.randn(M, N, device=dev)
    args = dict(act=kw.get("act", L.ACT_NONE), pA=kw.get("pA", 0.0), siteA=kw.get("siteA", 0), pB=kw.get("pB", 0.0), siteB=kw.get("siteB", 0), seed=5)
    for it in range(4):
        if it == 3:
            L.profile = {}
        ops.linear(x, w, b, residual=res, **args).backward(dy)
    prof = L.profile_collect()
    L.profile = None
    print("%-9s N=%-4d K=%-4d " % (name, N, K) + "  ".join("%s %.1f us" % (k.replace("rbm_linear_", ""), 1e3 * sum(ms for ms, _ in v)) for k, v in prof.items()))
