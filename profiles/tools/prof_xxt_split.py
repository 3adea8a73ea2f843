"""Time the track_C step at d = 100, k = 25, n = 20000 (fp32, codes given, so the step is the update, the products and the
blends): CUDA events over 200 steps after 20 warm-up steps.  With two library builds, alternates them in fresh processes:

    python profiles/tools/prof_xxt_split.py OLD.so NEW.so [rounds]

prints one line per run and the card's name and power limit."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def one():
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    from onmf_ontf_ndl_b200 import OnmfEngine, _lib
    d, k, n = 100, 25, 20000
    rng = np.random.default_rng(0)
    X = torch.from_numpy(rng.random((n, d))).cuda().float()
    H = torch.from_numpy(rng.random((n, k)) * (rng.random((n, k)) < 0.2)).cuda().float()
    eng = OnmfEngine(d, k, dtype=torch.float32, track_C=True)
    eng.set_state(rng.random((d, k)) / 10)
    for t in range(1, 21):
        eng.step(X, float(t), codes=H)
    eng.flush()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for t in range(21, 221):
        eng.step(X, float(t), codes=H)
    eng.flush()
    e1.record()
    torch.cuda.synchronize()
    C = eng.state()[3].double().cpu().numpy()
    print(json.dumps(dict(lib=_lib.LIB_PATH, ms_per_step=e0.elapsed_time(e1) / 200, C_sum=float(C.sum()))))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "one":
        one()
        sys.exit(0)
    libs, rounds = sys.argv[1:3], int(sys.argv[3]) if len(sys.argv) > 3 else 3
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True).stdout.strip())
    for _ in range(rounds):
        for lib in libs:
            env = dict(os.environ, ONMF_B200_LIB=os.path.abspath(lib))
            out = subprocess.run([sys.executable, os.path.abspath(__file__), "one"], env=env, capture_output=True, text=True)
            print(out.stdout.strip() or out.stderr[-2000:])
