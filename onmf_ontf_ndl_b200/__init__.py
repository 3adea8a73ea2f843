"""b200-onmf: B200-native online NMF / NTF dictionary learning behind the reference's
Online_NMF / Online_NTF API (HanbaekLyu/ONMF_ONTF_NDL src/onmf.py, src/ontf.py).

    from onmf_ontf_ndl_b200 import Online_NMF, Online_NTF, update_code_within_radius

Host code is Python; all arithmetic runs in libonmf_b200.so (hand-written sm_100a CUDA, C ABI in
include/onmf_b200.h).  There is no CPU fallback.
"""
from .onmf import Online_NMF, update_code_within_radius  # noqa: F401
from .ontf import Online_NTF  # noqa: F401
from .engine import OnmfEngine  # noqa: F401
from .reconstruct import reconstruct_from_patches_2d, reconstruct_image, reconstruct_network, \
    reconstruct_network_chains  # noqa: F401

__all__ = ["Online_NMF", "Online_NTF", "update_code_within_radius", "OnmfEngine", "reconstruct_image",
           "reconstruct_network", "reconstruct_network_chains", "reconstruct_from_patches_2d"]
