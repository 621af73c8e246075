# 04_find_contours.py -- drop-in SHIM for the reference's stage 04.  Both GPU-backed steps come from omni_b200.contours:
# `thinning_zhangsuen` (04_find_contours.py:35-99 of the reference, Zhang-Suen thinning of the edge planes) and
# `trace_centerlines` (04:101-205): connected components, degree maps and the walk along the skeleton in one call
# (omni_trace_centerlines), one component per CTA -- same polylines, same order, same log lines except the time-driven
# "visited" lines (tests/golden/trace.npz is frozen from the reference).  Everything else is the reference's own code: rename
# the reference's file to `04_find_contours_ref.py` (same directory) and put this file in its place -- it loads the original
# module, swaps the two functions and runs the original `vectorize_all`, so contours.pkl and the log are the reference's.
import importlib.util
import os
import sys

import _omni_path

_omni_path.add()
from omni_b200 import contours  # noqa: E402

_HERE = os.path.dirname(os.path.abspath(__file__))
_REF = os.path.join(_HERE, "04_find_contours_ref.py")


def _load_reference():
    if not os.path.exists(_REF):
        raise FileNotFoundError(f"{_REF} not found: rename the reference's 04_find_contours.py to 04_find_contours_ref.py "
                                "(this shim replaces only its thinning step)")
    spec = importlib.util.spec_from_file_location("find_contours_ref", _REF)
    mod = importlib.util.module_from_spec(spec)
    sys.modules["find_contours_ref"] = mod
    spec.loader.exec_module(mod)
    return mod


ref = _load_reference()
ref.thinning_zhangsuen = contours.thinning_zhangsuen          # same signature, same result, same progress lines
ref.trace_centerlines = contours.trace_centerlines            # same signature, same polylines, same progress lines
thinning_zhangsuen = contours.thinning_zhangsuen
trace_centerlines = contours.trace_centerlines
vectorize_layer = ref.vectorize_layer
vectorize_all = ref.vectorize_all
load_config = ref.load_config

if __name__ == "__main__":
    config = load_config()
    vectorize_all(config)
