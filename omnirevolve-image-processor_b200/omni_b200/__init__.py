"""omni_b200 -- B200-native stages 01_resize / 02_color_extract / 03_edge_detect of the
omnirevolve image pipeline.  Arithmetic runs in hand-written sm_100a CUDA kernels behind the C ABI
of include/omni_b200.h (csrc/, lib/libomni_b200.so); this package is the host-side mirror of the
reference's stage functions.  There is no CPU fallback."""
from .capi import OmniError, LIB_PATH  # noqa: F401
from .ops import Engine, EdgeConfig, TraceResult, get_engine, pinned_empty  # noqa: F401

__all__ = ["Engine", "EdgeConfig", "TraceResult", "get_engine", "pinned_empty", "OmniError", "LIB_PATH"]
