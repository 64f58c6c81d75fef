"""vsom-b200: the VSOM training / scoring hot path on B200, behind the C-ABI of include/vsom_b200.h.

This Python package is a thin ctypes binding of libvsom_b200.so for the tests and the bench harness; the
drop-in surface for users of the reference is the C++ class set in include/ (SOM.hpp, Transformation.hpp, ...)
implemented in host/ on top of the same C-ABI.  There is no CPU fallback: without the CUDA library or a
B200 every call fails loudly.
"""
from .binding import (  # noqa: F401
    CLR,
    CLUSTER_HITS,
    CLUSTER_UNIFORM,
    EXPONENTIAL,
    INVERSE_PROPORTIONAL,
    MEDIAN,
    ORDER_EIGEN_SSE,
    ORDER_LANES,
    ORDER_REFERENCE,
    STANDARD,
    VsomContext,
    VsomError,
    exported_symbols,
    lib,
    lib_path,
    model_length,
)
from .build import build  # noqa: F401
