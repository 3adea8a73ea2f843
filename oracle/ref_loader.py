"""Import the UNMODIFIED reference (HanbaekLyu/ONMF_ONTF_NDL) from a checkout named by ONMF_REFERENCE_ROOT.

TEST INFRASTRUCTURE ONLY.  The reference is not part of this repository; without
ONMF_REFERENCE_ROOT nothing here can load it.  Used by `oracle/make_golden.py` to generate
the committed fixtures under `tests/golden/` and by `tests/test_oracle_vs_reference.py`
(skipped when no reference checkout is named).

The reference imports three modules that are not installed here and that it never
uses arithmetically on the hot path (SURVEY.md §8c):
  * matplotlib / matplotlib.pyplot  (src/onmf.py:7, src/ontf.py:8  -- unused)
  * progressbar                     (src/ontf.py:6                 -- unused)
  * tensorly (unfold, tenalg.khatri_rao, decomposition.parafac; src/ontf.py:10-13)
    -- only `unfold` is called (src/ontf.py:204,207); its numpy-backend definition is
    reshape(moveaxis(t, mode, 0), (t.shape[mode], -1)).
They are stubbed in sys.modules before the import; nothing in the reference is edited.
"""
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("ONMF_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "src", "ontf.py"))


def _stub(name, **attrs):
    if name in sys.modules:
        return sys.modules[name]
    m = types.ModuleType(name)
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def _unfold(t, mode):
    return np.reshape(np.moveaxis(t, mode, 0), (t.shape[mode], -1))


def load_reference():
    """Returns (ref_onmf_module, ref_ontf_module)."""
    if not reference_available():
        raise RuntimeError("no reference checkout: set ONMF_REFERENCE_ROOT (now %r)" % REFERENCE_ROOT)
    try:
        import matplotlib.pyplot  # noqa: F401
    except Exception:
        mpl = _stub("matplotlib")
        mpl.pyplot = _stub("matplotlib.pyplot")
    try:
        import progressbar  # noqa: F401
    except Exception:
        _stub("progressbar")
    try:
        import tensorly  # noqa: F401
    except Exception:
        tl = _stub("tensorly", unfold=_unfold)
        tl.tenalg = _stub("tensorly.tenalg", khatri_rao=None)
        tl.decomposition = _stub("tensorly.decomposition", parafac=None)
    import importlib.util

    mods = []
    for nm in ("onmf", "ontf"):
        spec = importlib.util.spec_from_file_location(
            "_reference_src_" + nm, os.path.join(REFERENCE_ROOT, "src", nm + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mods.append(mod)
    return tuple(mods)


def load_reference_driver(name):
    """Import one of the reference's top-level driver scripts (e.g. "network_reconstruction_nx",
    "image_reconstruction_tensor") UNMODIFIED, bound to the reference's own `src` package.  Non-arithmetic imports that
    are not installed here (seaborn, matplotlib, skimage, progressbar, tensorly) are stubbed; `utils.onmf` / `utils.ontf`
    (a package the reference imports but does not ship, SURVEY.md §A.4) are aliased to its `src.onmf` / `src.ontf`."""
    import importlib
    import importlib.util
    onmf, ontf = load_reference()
    try:
        import matplotlib.image  # noqa: F401
    except Exception:
        sys.modules["matplotlib"].image = _stub("matplotlib.image")
    for nm in ("seaborn",):
        try:
            importlib.import_module(nm)
        except Exception:
            _stub(nm)
    try:
        import skimage.transform  # noqa: F401
    except Exception:
        sk = _stub("skimage")
        sk.transform = _stub("skimage.transform", downscale_local_mean=None)
    saved = {k: sys.modules.get(k) for k in ("src", "src.onmf", "src.ontf", "utils", "utils.onmf", "utils.ontf")}
    try:
        pkg = types.ModuleType("src"); pkg.__path__ = []
        upkg = types.ModuleType("utils"); upkg.__path__ = []
        pkg.onmf, pkg.ontf, upkg.onmf, upkg.ontf = onmf, ontf, onmf, ontf
        sys.modules.update({"src": pkg, "src.onmf": onmf, "src.ontf": ontf, "utils": upkg, "utils.onmf": onmf,
                            "utils.ontf": ontf})
        spec = importlib.util.spec_from_file_location("_reference_driver_" + name,
                                                      os.path.join(REFERENCE_ROOT, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod
