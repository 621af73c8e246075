"""Stage 04 trace_centerlines on the GPU (omni_trace_centerlines, csrc/trace.cu) against the golden polylines of the reference
(tests/golden/trace.npz) and against the host walk (`contours.trace_centerlines(..., maps=<cv2 maps>)`, itself pinned to the
golden set by test_contours_mirror.py): same polylines in the same order, the same log lines, cv2's component stats."""
import contextlib
import io
import os
import pickle
import re

import cv2
import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from helpers import blob_mask, synth

pytestmark = pytest.mark.gpu

Z = np.load(f"{GOLDEN}/trace.npz")
CASES = sorted(k[:-5] for k in Z.files if k.endswith("_skel"))


def _blank(log):
    return "\n".join(ln for ln in re.sub(r"[0-9.]+s", "Xs", log).splitlines() if "visited" not in ln)


def _maps(sk):
    S = (sk > 0).astype(np.uint8)
    k = np.ones((3, 3), np.uint8)
    k[1, 1] = 0
    deg = cv2.filter2D(S, cv2.CV_8U, k, borderType=cv2.BORDER_CONSTANT)
    return deg, (S == 1) & (deg == 1), (S == 1) & (deg >= 3)


def _host(sk, layer="L"):
    from omni_b200 import contours
    with contextlib.redirect_stdout(io.StringIO()) as log:
        paths = contours.trace_centerlines(sk, layer, maps=_maps(sk))
    return paths, log.getvalue()


def _same_paths(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.dtype == np.int32 and x.shape[1:] == (1, 2) and np.array_equal(x, y)


def _check_plane(r, sk):
    """One TraceResult against the host walk and cv2's stats."""
    _same_paths(r.paths, _host(sk)[0])
    num, _lab, st, _c = cv2.connectedComponentsWithStats((sk > 0).astype(np.uint8), connectivity=8)
    assert r.stats.shape == (num - 1, 5) and np.array_equal(r.stats, st[1:])
    assert r.total_fg == int((sk > 0).sum()) and int(r.polylines.sum()) == len(r.paths)


@pytest.fixture(scope="module")
def eng():
    import omni_b200
    return omni_b200.get_engine()


@pytest.mark.parametrize("case", CASES)
def test_gpu_trace_equals_reference_golden(case):
    from omni_b200 import contours
    sk = Z[case + "_skel"]
    with contextlib.redirect_stdout(io.StringIO()) as log:
        paths = contours.trace_centerlines(sk.copy(), case)
    assert [len(p) for p in paths] == Z[case + "_len"].tolist()
    assert all(p.dtype == np.int32 and p.shape[1:] == (1, 2) for p in paths)
    pts = np.concatenate([p.reshape(-1, 2) for p in paths]) if paths else np.zeros((0, 2), np.int32)
    assert np.array_equal(pts, Z[case + "_pts"])
    assert _blank(log.getvalue()) == str(Z[case + "_log"])


def test_gpu_trace_golden_all_planes_in_one_call(eng):
    """Every golden skeleton of one shape as planes of one call (the 192 x 256 and 128 x 192 sets)."""
    for shape in {Z[c + "_skel"].shape for c in CASES}:
        sks = [Z[c + "_skel"] for c in CASES if Z[c + "_skel"].shape == shape]
        for r, sk in zip(eng.host_trace_centerlines(np.stack(sks)), sks):
            _check_plane(r, sk)


def _thin(eng, planes):
    return eng.host_thin_zhangsuen(np.ascontiguousarray(planes, dtype=np.uint8))[0]


def _canny_skeletons(eng, h, w, n, seed):
    e = [cv2.Canny(cv2.GaussianBlur(blob_mask(h, w, seed + i, 0.2 + 0.1 * (i % 4), k=7), (3, 3), 0), 50, 150) for i in range(n)]
    return _thin(eng, np.stack(e))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_gpu_trace_canny_skeletons_vs_host(eng, seed):
    sks = _canny_skeletons(eng, 150 + 31 * seed, 201 + 17 * seed, 4, 10 * seed)
    for r, sk in zip(eng.host_trace_centerlines(sks), sks):
        _check_plane(r, sk)


@pytest.mark.parametrize("shape", [(60, 80), (33, 47), (1, 300), (300, 1), (2, 2), (7, 1), (1, 5), (65, 129)])
def test_gpu_trace_thick_random_vs_host(eng, shape):
    """Thick 35 % noise (junction-rich, wandering cycles that trip the guard) and thinned noise, odd and degenerate shapes."""
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    thick = (rng.random((3,) + shape) < 0.35).astype(np.uint8) * 255
    for planes in (thick, _thin(eng, thick)):
        for r, sk in zip(eng.host_trace_centerlines(planes), planes):
            _check_plane(r, sk)


def test_gpu_trace_dots_and_loops(eng):
    """Isolated pixels give no polyline; closed loops get the closing point."""
    sk = np.zeros((64, 96), np.uint8)
    sk[::7, ::5] = 255                                       # isolated pixels
    cv2.rectangle(sk, (3, 3), (40, 30), 255, 1)              # a 4-connected loop
    cv2.circle(sk, (70, 40), 15, 255, 1)                     # an 8-connected loop
    cv2.line(sk, (50, 5), (90, 20), 255, 1)                  # an open path with two endpoints
    r = eng.host_trace_centerlines(sk)[0]
    _check_plane(r, sk)
    closed = [p for p in r.paths if np.array_equal(p[0], p[-1])]
    assert len(closed) >= 2 and min(len(p) for p in r.paths) >= 2


def test_gpu_trace_components_touching_every_border(eng):
    sk = np.zeros((50, 70), np.uint8)
    sk[0, :] = sk[-1, :] = sk[:, 0] = sk[:, -1] = 255        # a frame on the border
    cv2.line(sk, (0, 25), (35, 40), 255, 1)                  # a path leaving the frame
    sk[10, 10] = sk[49, 35] = 255
    noise = (np.random.default_rng(3).random(sk.shape) < 0.3).astype(np.uint8) * 255
    noise[5:-5, 5:-5] = 0                                    # noise along every border
    for plane in (sk, noise, _thin(eng, noise[None])[0]):
        _check_plane(eng.host_trace_centerlines(plane)[0], plane)


def test_gpu_trace_large_components_global_path(eng):
    """Components whose bounding box (plus a frame) exceeds the 200 KB shared-memory window walk from global memory: a frame on
    the border of a 700 x 900 plane with paths and loops attached, a long chain across the plane, and small components beside
    them in the same call (shared-memory path)."""
    h, w = 700, 900
    a = np.zeros((h, w), np.uint8)
    a[0, :] = a[-1, :] = a[:, 0] = a[:, -1] = 255
    for i in range(12):
        cv2.line(a, (0, 40 + 50 * i), (200 + 40 * i, 90 + 45 * i), 255, 1)
    cv2.circle(a, (600, 300), 120, 255, 1)
    cv2.line(a, (480, 300), (300, 300), 255, 1)
    b = np.zeros((h, w), np.uint8)
    pts = np.random.default_rng(7).integers(5, [w - 5, h - 5], (40, 2)).astype(np.int32)
    cv2.polylines(b, [pts], False, 255, 1)                    # one long, self-crossing chain across the plane
    b[::37, ::41] = 255
    c = _canny_skeletons(eng, h, w, 1, 40)[0]
    planes = np.stack([a, b, c])
    bb = [cv2.connectedComponentsWithStats((p > 0).astype(np.uint8), connectivity=8)[2][1:] for p in planes]
    assert all(((s[:, 2] + 2) * (s[:, 3] + 2) > 200 * 1024).any() for s in bb[:2])
    for r, sk in zip(eng.host_trace_centerlines(planes), planes):
        _check_plane(r, sk)


def test_gpu_trace_empty_planes_in_one_call(eng):
    sks = _canny_skeletons(eng, 90, 130, 2, 60)
    z = np.zeros_like(sks[0])
    planes = np.stack([z, sks[0], z, z, sks[1], z])
    res = eng.host_trace_centerlines(planes)
    assert len(res) == 6
    for r, sk in zip(res, planes):
        _check_plane(r, sk)
    assert res[0].paths == [] and res[0].total_fg == 0 and res[0].stats.shape == (0, 5)
    allz = eng.host_trace_centerlines(np.zeros((3, 5, 7), np.uint8))
    assert all(r.paths == [] and r.total_fg == 0 for r in allz)


def test_gpu_trace_device_and_host_forms_agree_on_strided_views(eng):
    import torch
    sks = _canny_skeletons(eng, 120, 170, 3, 80)
    buf = torch.zeros((5, 140, 200), dtype=torch.uint8, device="cuda")
    buf[1:4, 7:127, 11:181] = torch.from_numpy(sks).cuda()
    view = buf[1:4, 7:127, 11:181]                           # plane stride 28000, pitch 200, offset start
    dev = eng.trace_centerlines(view)
    host_buf = np.zeros((5, 140, 200), np.uint8)
    host_buf[1:4, 7:127, 11:181] = sks
    host = eng.host_trace_centerlines(host_buf[1:4, 7:127, 11:181])
    for d, hst, sk in zip(dev, host, sks):
        _same_paths(d.paths, hst.paths)
        assert np.array_equal(d.stats, hst.stats) and np.array_equal(d.polylines, hst.polylines) and d.total_fg == hst.total_fg
        _check_plane(d, sk)
    inv = eng.host_trace_centerlines((sks[:, ::-1, :] > 0))  # negative pitch and a bool array: copied, same result
    for r, sk in zip(inv, sks):
        _check_plane(r, np.ascontiguousarray(sk[::-1]))


def test_gpu_trace_4096_k8_edges(eng):
    """A 4096^2, K=8 edge set from omni_color_edge, thinned on the device, traced in one call; the two smallest layers (by skeleton
    pixels) compared exactly with the host walk, every layer's stats with cv2's."""
    import torch
    from omni_b200 import EdgeConfig
    img = torch.from_numpy(synth(4096, 4096, 3, cell=64)).cuda()
    ctr = np.array([[25 + 30 * i, 100 + 8 * i, 160 - 7 * i] for i in range(8)], np.float32)
    _l, _m, edges = eng.color_edge(img, ctr, np.arange(8, dtype=np.uint8), EdgeConfig())
    skel = eng.thin_zhangsuen(edges)
    res = eng.trace_centerlines(skel)
    sks = skel.cpu().numpy()
    for r, sk in zip(res, sks):
        num, _lab, st, _c = cv2.connectedComponentsWithStats((sk > 0).astype(np.uint8), connectivity=8)
        assert np.array_equal(r.stats, st[1:]) and r.total_fg == int((sk > 0).sum())
    order = sorted((i for i in range(8) if res[i].total_fg > 0), key=lambda i: res[i].total_fg)
    assert len(order) >= 2
    for i in order[:2]:
        _same_paths(res[i].paths, _host(sks[i])[0])


def test_stage04_shim_contours_pkl_equals_host_walk(tmp_path, eng):
    """The stage-04 shim at 1024^2, K=4: a stand-in for the reference's file whose `vectorize_all` traces every layer's skeleton
    and pickles the polylines as contours.pkl; the bytes equal those of the same pickle made with the host walk."""
    import shutil
    import subprocess
    import sys
    from omni_b200 import EdgeConfig
    src = os.path.join(ROOT, "omnirevolve-image-processor_b200", "image_processor")
    for f in ("04_find_contours.py", "_omni_path.py"):
        shutil.copy(os.path.join(src, f), tmp_path / f)
    (tmp_path / "04_find_contours_ref.py").write_text(
        "import os, pickle, cv2\n"
        "def load_config():\n"
        "    class C: pass\n"
        "    c = C(); c.output_dir = os.environ['OUT_DIR']; c.color_names = ['l0', 'l1', 'l2', 'l3']; return c\n"
        "def thinning_zhangsuen(img, layer):\n"
        "    raise RuntimeError('the CPU thinning must have been replaced')\n"
        "def trace_centerlines(skel, layer):\n"
        "    raise RuntimeError('the per-component tracing must have been replaced')\n"
        "def vectorize_layer(name, cfg):\n"
        "    e = cv2.imread(os.path.join(cfg.output_dir, name, 'edges.png'), cv2.IMREAD_GRAYSCALE)\n"
        "    return name, trace_centerlines(thinning_zhangsuen(e, layer=name), layer=name)\n"
        "def vectorize_all(cfg):\n"
        "    out = dict(vectorize_layer(n, cfg) for n in cfg.color_names)\n"
        "    pickle.dump(out, open(os.path.join(cfg.output_dir, 'contours.pkl'), 'wb'))\n")
    ctr = np.array([[40, 128, 128], [110, 140, 120], [160, 120, 150], [220, 128, 128]], np.float32)
    edges = eng.host_color_edge(synth(1024, 1024, 0), ctr, np.arange(4, dtype=np.uint8), EdgeConfig())["edges"]
    out = tmp_path / "out"
    want = {}
    for i in range(4):
        os.makedirs(out / f"l{i}")
        cv2.imwrite(str(out / f"l{i}" / "edges.png"), edges[i])
    sks = _thin(eng, edges)
    for i in range(4):
        want[f"l{i}"] = _host(sks[i], f"l{i}")[0]
    env = dict(os.environ, OUT_DIR=str(out), OMNI_B200_HOME=os.path.join(ROOT, "omnirevolve-image-processor_b200"))
    r = subprocess.run([sys.executable, str(tmp_path / "04_find_contours.py")], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:]
    assert sum(len(v) for v in want.values()) > 0
    assert (out / "contours.pkl").read_bytes() == pickle.dumps(want)
    for n, v in want.items():
        assert f"[{n}] Trace done: {len(v)} polylines" in r.stdout
