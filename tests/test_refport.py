"""oracle/refport.py must compute what the reference's own functions compute: checked against outputs of the unmodified
reference frozen under tests/golden/ (tools/make_golden.py, tools/make_golden_process_colors.py).  The stage-04 swap-point
test imports the reference module itself and runs only when OMNI_REFERENCE_DIR names it."""
import importlib.util
import json
import os
import sys

import cv2
import numpy as np
import pytest

from conftest import GOLDEN, REFERENCE_DIR
from oracle import refport as rp
from helpers import PIPE_CASES, load_pipe_case


def _load(fname, modname):
    sys.dont_write_bytecode = True
    if REFERENCE_DIR not in sys.path:
        sys.path.append(REFERENCE_DIR)          # for `from config import ...`
    spec = importlib.util.spec_from_file_location(modname, os.path.join(REFERENCE_DIR, fname))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_kmeans_lab_and_assign():
    """02:32-56 in a fresh process (centres, raw labels) and 02:17-23 (layer names by darkness rank -> cluster index) against
    the centres, labels and palette_by_name.json frozen from the reference on the pipeline cases (K = 4, 4, 8)."""
    for case in PIPE_CASES:
        z, meta = load_pipe_case(case)
        names = meta["names"]
        c = rp.kmeans_lab_centers(z["resized"], len(names))
        assert np.array_equal(c, z["centers"]), case
        assert np.array_equal(rp.assign_lab(z["resized"], c), z["labels"]), case
        assert np.array_equal(rp.assign_lab_chunked(z["resized"], c, rows=37), z["labels"]), case
        ranked = sorted(names, key=rp.darkness_rank)
        assert [ranked.index(n) for n in names] == [meta["palette_by_name"][n]["cluster_index"] for n in names], case


def test_assign_labels_rgb():
    """process_colors.py:69-77 (int16 wrap) against the label maps the reference CLI saved (K = 5, analyzer and eight palettes)."""
    z = np.load(os.path.join(GOLDEN, "process_colors.npz"))
    meta = json.load(open(os.path.join(GOLDEN, "process_colors.json")))
    rgb = cv2.cvtColor(z["input"], cv2.COLOR_BGR2RGB)
    for case in ("adaptive5", "analyzer", "eight"):
        pal = np.array([c["rgb"] for c in meta[case]["palette"]["colors"]], np.uint8)
        assert np.array_equal(rp.assign_labels_rgb(rgb, pal), z[f"labels_{case}"]), case


def test_edge_layer_and_resize():
    """01_resize.py:7-23 against the reference's resize_if_needed on its 2:1, 3:1, fractional and no-op paths
    (functions.npz), and 03_edge_detect.py:13-40 against the edge planes its stage 03 wrote for the pipeline cases
    (blur 3 / 7 / 5, Canny 50/150, 22/70, 100/200)."""
    f = np.load(os.path.join(GOLDEN, "functions.npz"))
    for tag in ("rz_2to1", "rz_3to1", "rz_frac", "rz_frac2", "rz_noop"):
        assert np.array_equal(rp.resize_if_needed(f[tag + "_src"], int(f[tag + "_md"])), f[tag + "_dst"]), tag
    for case in PIPE_CASES:
        z, meta = load_pipe_case(case)
        cfg = meta["config"]
        for m, e in zip(z["masks"], z["edges"]):
            assert np.array_equal(rp.edge_layer(m, cfg["edge_low_threshold"], cfg["edge_high_threshold"], cfg["edge_kernel_size"]), e), case


def test_skeleton_degree_global_equals_per_component():
    """The one-shot degree map equals the reference's per-component maps on skeleton pixels (04:113-125)."""
    from helpers import blob_mask
    from oracle import cmodel as cm
    for seed in (1, 2):
        sk = cm.thin_zhangsuen(blob_mask(90, 140, seed, 0.45, k=5))
        deg, ep, jn = rp.skeleton_degree(sk)
        deg_c, ep_c, jn_c = rp.skeleton_degree_per_component(sk)
        on = sk > 0
        assert np.array_equal(deg[on], deg_c[on]) and np.array_equal(ep, ep_c) and np.array_equal(jn, jn_c)
        assert ep.any() or jn.any()


@pytest.mark.reference
def test_stage04_swap_point_with_real_reference(tmp_path):
    """The stage-04 shim (image_processor/04_find_contours.py) replaces ONE module global of the reference's stage 04.
    With the real reference file: the names the shim relies on exist, `vectorize_layer` resolves `thinning_zhangsuen`
    through the module globals, and a skeleton that equals the reference's (here from the pinned C oracle -- the GPU
    kernel is checked against the same oracle) yields the reference's contours.pkl byte for byte."""
    import contextlib
    import io
    import pickle
    from oracle import cmodel as cm
    from helpers import blob_mask
    ref = _load("04_find_contours.py", "ref_fc_swap")
    for name in ("thinning_zhangsuen", "trace_centerlines", "vectorize_layer", "vectorize_all", "load_config"):
        assert callable(getattr(ref, name)), name

    class Cfg:
        pass
    cfg = Cfg()
    cfg.output_dir = str(tmp_path)
    cfg.color_names = ["layer_a"]
    os.makedirs(tmp_path / "layer_a")
    edges = cv2.Canny(cv2.GaussianBlur(blob_mask(60, 80, 3, 0.4, k=7), (3, 3), 0), 50, 150)
    cv2.imwrite(str(tmp_path / "layer_a" / "edges.png"), edges)
    with contextlib.redirect_stdout(io.StringIO()):
        ref.vectorize_all(cfg)
    want = pickle.load(open(tmp_path / "layer_a" / "contours.pkl", "rb"))
    calls = []

    def swapped(bin_0_255, layer):
        calls.append(layer)
        return cm.thin_zhangsuen(bin_0_255)
    ref.thinning_zhangsuen = swapped
    with contextlib.redirect_stdout(io.StringIO()):
        ref.vectorize_all(cfg)
    got = pickle.load(open(tmp_path / "layer_a" / "contours.pkl", "rb"))
    assert calls == ["layer_a"]
    assert len(got) == len(want) and all(np.array_equal(a, b) for a, b in zip(got, want))
