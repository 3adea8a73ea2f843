"""fp32 production engine free-running on the full_cfg5 fixture next to the fp64 engine: per-step code / W / A / B errors
(where does the fp32 dictionary error at the benchmarked shape come from).  GPU only; analysis tool."""
import os
import sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np
import torch
from onmf_ontf_ndl_b200 import OnmfEngine, _lib

g = np.load(os.path.join(ROOT, "tests", "golden", "full_cfg5.npz"))
ntr, k = int(g["n_train"]), int(g["k"])
X = np.random.RandomState(int(g["x_seed"])).rand(1024, ntr + int(g["n_holdout"]))
W0 = np.random.RandomState(int(g["seed"])).rand(1024, k)
dev = torch.device("cuda", 0)
use_tc = os.environ.get("DIAG_TC", "1") == "1"
pool64 = torch.from_numpy(np.ascontiguousarray(X[:, :ntr].T)).to(dev)
pool32 = pool64.float().contiguous()
e64 = OnmfEngine(1024, k, alpha=1.0, dtype=torch.float64, device=dev)
e32 = OnmfEngine(1024, k, alpha=1.0, dtype=torch.float32, device=dev, use_tc=use_tc, collect_stats=True)
e64.set_state(W0); e32.set_state(W0)
nb = g["idx"].shape[1]
x64 = torch.empty(nb, 1024, dtype=torch.float64, device=dev); x32 = torch.empty(nb, 1024, dtype=torch.float32, device=dev)
rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm())
pa = lambda a, b: float(((a.double() - b.double()).norm(dim=0) / b.double().norm(dim=0)).max())
for i in range(int(g["iters"])):
    idx = torch.from_numpy(g["idx"][i].astype(np.int64)).to(dev)
    _lib.gather_rows(pool64, idx, x64); _lib.gather_rows(pool32, idx, x32)
    H64 = e64.step(x64, float(i + 1)).clone(); H32 = e32.step(x32, float(i + 1)).clone()
    W6, A6, B6, _ = e64.state(); W3, A3, B3, _ = e32.state()
    torch.cuda.synchronize()
    Href = torch.from_numpy(g["H_%d" % i]).to(dev)
    if os.environ.get("DIAG_COLS", "1") == "1":
        ce = (H32.double() - Href).norm(dim=1) / Href.norm(dim=1).clamp_min(1e-30)
        top = torch.topk(ce, 4)
        tot2 = float(((H32.double() - Href) ** 2).sum())
        for j, v in zip(top.indices.tolist(), top.values.tolist()):
            s32 = set(torch.nonzero(H32[j]).flatten().tolist()); sr = set(torch.nonzero(Href[j]).flatten().tolist())
            share = float(((H32[j].double() - Href[j]) ** 2).sum()) / max(tot2, 1e-300)
            print("    col %5d rel %.2e share-of-err %.2f nnz32 %d nnzref %d only32 %s onlyref %s" %
                  (j, v, share, len(s32), len(sr), sorted(s32 - sr)[:6], sorted(sr - s32)[:6]))
        print("    median col err %.2e  90%% %.2e  99%% %.2e" % tuple(float(torch.quantile(ce, q)) for q in (0.5, 0.9, 0.99)))
    print("step %2d codes32-vs-ref %.2e codes64-vs-ref %.2e | W per-atom %.2e  A %.2e  B %.2e | stats %s"
          % (i, rel(H32, Href), rel(H64, Href), pa(W3, W6), rel(A3, A6), rel(B3, B6),
             {k_: v for k_, v in e32.read_stats().items() if k_ in ("overflow", "flagged", "max_active")}), flush=True)
Wref = torch.from_numpy(g["W"]).to(dev)
print("final per-atom fp32 vs reference %.3e   fp64 vs reference %.3e" % (pa(W3, Wref), pa(W6, Wref)))

# ---- E2: fp32 aggregation + dictionary update with the fp64 engine's codes (isolates the coder from the rest) ----
e64 = OnmfEngine(1024, k, alpha=1.0, dtype=torch.float64, device=dev)
e32 = OnmfEngine(1024, k, alpha=1.0, dtype=torch.float32, device=dev, use_tc=use_tc)
e64.set_state(W0); e32.set_state(W0)
for i in range(int(g["iters"])):
    idx = torch.from_numpy(g["idx"][i].astype(np.int64)).to(dev)
    _lib.gather_rows(pool64, idx, x64); _lib.gather_rows(pool32, idx, x32)
    H64 = e64.step(x64, float(i + 1)).clone()
    e32.step(x32, float(i + 1), codes=H64.float().contiguous())
    W6, A6, B6, _ = e64.state(); W3, A3, B3, _ = e32.state()
    torch.cuda.synchronize()
    err = ((W3.double() - W6).norm(dim=0) / W6.norm(dim=0))
    top = torch.topk(err, 3)
    print("E2 step %2d W per-atom %.2e  A %.2e  B %.2e | worst atoms %s err %s A_jj %s" %
          (i, float(err.max()), rel(A3, A6), rel(B3, B6), top.indices.tolist(), ["%.1e" % v for v in top.values.tolist()],
           ["%.2e" % float(A6[j, j]) for j in top.indices.tolist()]), flush=True)
print("A_jj quantiles", np.quantile(np.diag(A6.cpu().numpy()), [0, 0.01, 0.1, 0.5, 0.9, 1.0]))
