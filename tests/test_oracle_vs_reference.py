"""The committed fixtures against the LIVE reference: regenerate a few of them with the unmodified reference
(a checkout named by ONMF_REFERENCE_ROOT, imported through oracle/ref_loader.py) and require bit-equality with what
is in tests/golden/.

The reference is not part of this repository: without ONMF_REFERENCE_ROOT these tests skip, and the fixtures they
guard are checked by tests/test_oracle.py and tests/test_gpu_parity.py.  CPU only.
ONMF_SLOW=1 additionally regenerates the full-length cfg1 and cfg5 runs (~1 + ~2 CPU-minutes)."""
import os
import warnings

import numpy as np
import pytest

from oracle.ref_loader import reference_available

warnings.filterwarnings("ignore")
pytestmark = pytest.mark.skipif(not reference_available(), reason="no reference checkout (set ONMF_REFERENCE_ROOT)")

# scalars computed through BLAS reductions may differ in the last bit with the thread count
LOOSE = {"recon": 1e-12}


def _same(a, b, name):
    assert sorted(a.files) == sorted(b.files), name
    for k in a.files:
        x, y = a[k], b[k]
        if k in LOOSE:
            assert abs(float(x) - float(y)) <= LOOSE[k] * max(1.0, abs(float(y))), (name, k)
        else:
            assert x.shape == y.shape and np.array_equal(x, y), (name, k)


@pytest.mark.parametrize("names", [("cfg3_binary_motif", "cfg5_synthetic", "pgd_coder", "network_recons", "driver_tensor")])
def test_fixtures_regenerate_bit_identically(golden_dir, tmp_path, names):
    from oracle import make_golden
    make_golden.main(which=names, out_dir=str(tmp_path))
    for nm in names:
        _same(np.load(os.path.join(golden_dir, nm + ".npz")), np.load(os.path.join(str(tmp_path), nm + ".npz")), nm)


@pytest.mark.skipif(os.environ.get("ONMF_SLOW") != "1", reason="set ONMF_SLOW=1 (about 3 CPU-minutes)")
def test_full_length_fixtures_regenerate(golden_dir, tmp_path):
    from oracle import make_golden_full
    make_golden_full.OUT = str(tmp_path)
    make_golden_full.main(["cfg1", "cfg5"])
    for nm in ("full_cfg1", "full_cfg5"):
        _same(np.load(os.path.join(golden_dir, nm + ".npz")), np.load(os.path.join(str(tmp_path), nm + ".npz")), nm)
