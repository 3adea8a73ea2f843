"""bench.py --dump-outputs: the arrays of the last timed step, identical from run to run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg1", "--steps", str(steps),
                        "--warmup", "5", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == steps
    return {nm[:-4]: np.load(os.path.join(str(out_dir), nm)) for nm in sorted(os.listdir(str(out_dir)))}


@pytest.mark.gpu
def test_dump_outputs_repeat_and_follow_steps(tmp_path):
    a = _bench(tmp_path / "a", 3)
    b = _bench(tmp_path / "b", 3)
    c = _bench(tmp_path / "c", 4)
    d, k, n = 100, 25, 1000                                  # cfg1: every code row fits the sample
    assert {nm: x.shape for nm, x in a.items()} == {"codes": (n, k), "W": (d, k), "A": (k, k), "B": (k, d)}
    for nm, x in a.items():
        assert x.dtype == np.float32 and np.all(np.isfinite(x)), nm
        assert np.array_equal(x, b[nm]), nm
    assert a["codes"].min() >= 0 and a["codes"].max() > 0
    assert np.all(np.linalg.norm(a["W"], axis=0) <= 1 + 1e-5)
    assert not np.array_equal(a["W"], c["W"])                # one more timed step, one more dictionary update
