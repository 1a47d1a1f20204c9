"""pcb200 -- B200-native hot path of Epsilon-79th/linear-eigenvalue-problems-in-photonic-crystals (paper_2).

The sub-modules carry the reference's module names (environment, dielectric, discretization, pcfft,
orthogonalization, lobpcg, numerical_experiments) and public functions; the O(N^3) work runs in
csrc/libpcb200.so (hand-written sm_100a CUDA behind the C ABI of include/pcb200.h, called through
ctypes).  Import with

    import importlib; pcb = importlib.import_module("linear-eigenvalue-problems-in-photonic-crystals_b200")

and, to run scripts written against the reference's flat modules unchanged, ``pcb.install_as_reference_modules()``.
"""
import sys as _sys

from . import _lib, devarray, environment, dielectric, discretization, dispersion, pcfft, orthogonalization, lobpcg, numerical_experiments, sharded  # noqa: F401,E501
from .devarray import Context, DeviceBlock, get_context, pinned_empty, set_device  # noqa: F401
from ._lib import PcbError, backend  # noqa: F401

REFERENCE_MODULES = ("environment", "dielectric", "discretization", "pcfft", "orthogonalization", "lobpcg",
                     "numerical_experiments")


def install_as_reference_modules():
    """Register the sub-modules under the reference's flat names (``import lobpcg`` ...)."""
    me = _sys.modules[__name__]
    for name in REFERENCE_MODULES:
        _sys.modules[name] = getattr(me, name)
