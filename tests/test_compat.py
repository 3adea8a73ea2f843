"""The reference's drivers import `src.onmf`, `utils.onmf`, `utils.ontf`; compat/ provides those paths."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_driver_import_paths_and_constructor_forms():
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    try:
        for m in ("src", "src.onmf", "src.ontf", "utils", "utils.onmf", "utils.ontf"):
            sys.modules.pop(m, None)
        from src.onmf import Online_NMF, update_code_within_radius            # image_reconstruction.py:1
        from utils.onmf import Online_NMF as NMF2                              # ising_reconstruction.py:1
        from utils.ontf import Online_NTF                                      # image_reconstruction_tensor.py:1
        import onmf_ontf_ndl_b200 as pkg
        assert Online_NMF is pkg.Online_NMF and NMF2 is pkg.Online_NMF and Online_NTF is pkg.Online_NTF
        assert update_code_within_radius is pkg.update_code_within_radius
        X = np.random.rand(12, 30)
        a = Online_NMF(X, 5, 7, 3)                                            # image_reconstruction.py:349 positional form
        assert (a.n_components, a.iterations, a.batch_size) == (5, 7, 3) and a.code.shape == (5, 30)
        b = Online_NMF(X)                                                      # ising_reconstruction.py:194
        assert b.n_components == 100 and b.history == 0 and b.subsample is False
        c = Online_NMF(X, n_components=4, iterations=3, batch_size=2, ini_dict=None, ini_A=None, ini_B=None, ini_C=None,
                       history=0, alpha=None, beta=0.5)                        # ising_reconstruction.py:116-126
        assert c.beta == 0.5 and c._alpha() == 2                                # lasso_lars coder: alpha=None -> 2
        t = Online_NTF(np.random.rand(9, 3, 20), 6, iterations=4, sub_iterations=2, learn_joint_dict=True, mode=2,
                       batch_size=5)                                           # image_reconstruction_tensor.py:234-239
        assert t.code.shape == (3, 6) and t._alpha() == 2 and t.subsample is True
    finally:
        sys.path.remove(os.path.join(ROOT, "compat"))
        for m in ("src", "src.onmf", "src.ontf", "utils", "utils.onmf", "utils.ontf"):
            sys.modules.pop(m, None)


# ---------------------------------------------------------------------------------------------- a reference driver, end to end
import contextlib
import tempfile

import pytest


@contextlib.contextmanager
def _shim_on_path():
    """what a user of the reference does: put compat/ first on sys.path so that `utils.ontf` / `src.onmf` resolve here"""
    sys.path.insert(0, os.path.join(ROOT, "compat"))
    mods = ("src", "src.onmf", "src.ontf", "utils", "utils.onmf", "utils.ontf")
    for m in mods:
        sys.modules.pop(m, None)
    try:
        yield
    finally:
        sys.path.remove(os.path.join(ROOT, "compat"))
        for m in mods:
            sys.modules.pop(m, None)


def _per_atom(W, Wref):
    return float(np.max(np.linalg.norm(W - Wref, axis=0) / np.maximum(np.linalg.norm(Wref, axis=0), 1e-30)))


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp64", 1e-8), ("fp32", 1e-3)])
def test_tensor_driver_call_sequence_through_shim(golden_dir, monkeypatch, precision, tol):
    """Image_Reconstructor_tensor.train_dict (reference image_reconstruction_tensor.py:220-262) as a user of the shim runs
    it: `from utils.ontf import Online_NTF`, per epoch `extract_random_patches` (:87-124, np.random.choice per corner) then
    Online_NTF(X, r, iterations=sub_iterations, sub_iterations=block_iterations, learn_joint_dict, mode, batch_size
    [, ini_dict, ini_A, ini_B, history]).train_dict_single().  The driver file itself cannot travel to the GPU box, so
    its call sequence is restated here line by line; the expected dictionary is what the UNMODIFIED driver produced with
    the reference's own Online_NTF under the same seed (fixture driver_tensor, oracle/make_golden.py)."""
    from onmf_ontf_ndl_b200 import _host
    monkeypatch.setattr(_host, "DEFAULT_PRECISION", precision)
    g = np.load(os.path.join(golden_dir, "driver_tensor.npz"))
    data = g["img_u8"] / 255                                                   # read_img_as_array :77-82
    k, r = int(g["patch_size"]), int(g["n_components"])
    with _shim_on_path():
        from utils.ontf import Online_NTF                                      # :1
        np.random.seed(int(g["seed"]))
        W, At, Bt, ntf = None, [], [], None
        for t in np.arange(int(g["iterations"])):                              # :231
            x = data.shape                                                     # extract_random_patches :94-112
            X = np.zeros(shape=(k ** 2, 3, 1))
            for i in np.arange(int(g["num_patches"])):
                a = np.random.choice(x[0] - k)
                b = np.random.choice(x[1] - k)
                Y = data[a:a + k, b:b + k, :].reshape(k ** 2, 3, 1)
                X = Y if i == 0 else np.append(X, Y, axis=2)
            if t == 0:                                                         # :233-240
                ntf = Online_NTF(X, r, iterations=int(g["sub_iterations"]), sub_iterations=20,
                                 learn_joint_dict=bool(g["joint"]), mode=int(g["mode"]), batch_size=int(g["batch_size"]))
                W, At, Bt, H = ntf.train_dict_single()
            else:                                                              # :241-254
                ntf = Online_NTF(X, r, iterations=int(g["sub_iterations"]), sub_iterations=20,
                                 batch_size=int(g["batch_size"]), ini_dict=W, ini_A=At, ini_B=Bt,
                                 learn_joint_dict=bool(g["joint"]), mode=int(g["mode"]), history=ntf.history)
                W, At, Bt, H = ntf.train_dict_single()
    assert W.shape == g["W"].shape and W.dtype == np.float64
    assert W.min() >= 0 and np.all(np.linalg.norm(W, axis=0) <= 1 + 1e-6)      # SURVEY §4 invariants
    assert float(ntf.history) == float(g["history"])
    assert _per_atom(W, g["W"]) < tol


@pytest.mark.gpu
def test_reference_tensor_driver_runs_unmodified_on_the_shim(golden_dir, monkeypatch):
    """The UNMODIFIED driver file executed against compat/ (needs both a GPU and a reference checkout named by
    ONMF_REFERENCE_ROOT; skipped otherwise)."""
    ref = os.environ.get("ONMF_REFERENCE_ROOT", "")
    if not ref or not os.path.isfile(os.path.join(ref, "image_reconstruction_tensor.py")):
        pytest.skip("no reference checkout (set ONMF_REFERENCE_ROOT)")
    import importlib.util
    import types
    from PIL import Image
    from onmf_ontf_ndl_b200 import _host
    monkeypatch.setattr(_host, "DEFAULT_PRECISION", "fp64")
    g = np.load(os.path.join(golden_dir, "driver_tensor.npz"))
    for nm in ("matplotlib", "matplotlib.pyplot", "skimage", "skimage.transform"):
        if nm not in sys.modules:
            try:
                __import__(nm)
            except Exception:
                monkeypatch.setitem(sys.modules, nm, types.ModuleType(nm))
    if not hasattr(sys.modules["skimage.transform"], "downscale_local_mean"):
        sys.modules["skimage.transform"].downscale_local_mean = None
    cwd = os.getcwd()
    with _shim_on_path(), tempfile.TemporaryDirectory() as tmp:
        os.makedirs(os.path.join(tmp, "Image_dictionary"))
        Image.fromarray(g["img_u8"]).save(os.path.join(tmp, "crop.png"))
        spec = importlib.util.spec_from_file_location("_ref_driver_tensor", os.path.join(ref, "image_reconstruction_tensor.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        import onmf_ontf_ndl_b200 as pkg
        assert mod.Online_NTF is pkg.Online_NTF
        os.chdir(tmp)
        try:
            np.random.seed(int(g["seed"]))
            drv = mod.Image_Reconstructor_tensor(path="crop.png", n_components=int(g["n_components"]),
                                                 iterations=int(g["iterations"]), sub_iterations=int(g["sub_iterations"]),
                                                 batch_size=int(g["batch_size"]), num_patches=int(g["num_patches"]),
                                                 patch_size=int(g["patch_size"]), is_color=True)
            W = drv.train_dict(mode=int(g["mode"]), learn_joint_dict=bool(g["joint"]))
        finally:
            os.chdir(cwd)
    assert _per_atom(W, g["W"]) < 1e-8 and float(drv.ntf.history) == float(g["history"])
