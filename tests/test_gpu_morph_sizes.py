"""Stage-03 morphology for every edge_morph_kernel in 1..255 and any open / close count (03_edge_detect.py:23-30 passes the
config.json keys straight to cv2.getStructuringElement(MORPH_ELLIPSE) / cv2.morphologyEx).  The oracle is oracle.refport.edge_layer,
i.e. cv2 itself; every comparison is bit for bit.  Needs a B200: `-m gpu`."""
import json
import os
import subprocess
import sys

import cv2
import numpy as np
import pytest

from helpers import PIPE_CASES, load_pipe_case, synth, smooth_u8, blob_mask

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCRIPTS = os.path.join(ROOT, "omnirevolve-image-processor_b200", "image_processor")

SIZES = [2, 4, 5, 7, 8, 9, 10, 15, 16, 31, 33, 64, 127, 254, 255]
ITERS = [(1, 1), (0, 3), (2, 0), (2, 2)]
SHAPES = [(67, 93), (1, 200), (200, 1), (3, 300), (513, 1027)]
FAMILIES = [(1, "fast"), (0, "generic")]


@pytest.fixture(scope="module")
def eng():
    import omni_b200
    e = omni_b200.Engine(0)
    yield e
    e.set_fast_path(True)
    e.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


def _rp():
    from oracle import refport
    return refport


def _want(masks, ec):
    rp = _rp()
    return np.stack([rp.edge_layer(m, ec.low, ec.high, ec.ksize, ec.morph_k, ec.open_iters, ec.close_iters) for m in masks])


def _masks(h, w, seed):
    return np.stack([blob_mask(h, w, seed + s, p, k=5) for s, p in ((0, 0.5), (1, 0.25))])


def _centres(img, K):
    rp = _rp()
    ctr = rp.kmeans_lab_centers(img, K)
    _o, lut = rp.darkness_order(ctr)
    return ctr, lut.astype(np.uint8)


@pytest.mark.parametrize("hw", SHAPES, ids=[f"{h}x{w}" for h, w in SHAPES])
@pytest.mark.parametrize("mk", SIZES)
def test_binary_masks_every_size(eng, mk, hw):
    """Binary masks: bytes -> bits -> ELLIPSE kernel -> bit-plane edges (ksize 3, 7) or generic blur / Canny (ksize 9); both families."""
    import omni_b200
    masks = _masks(hw[0], hw[1], mk)
    d = dev(masks)
    for oi, ci in ITERS:
        for ks in (3, 7, 9):
            ec = omni_b200.EdgeConfig(low=50, high=150, ksize=ks, morph_k=mk, open_iters=oi, close_iters=ci)
            want = _want(masks, ec)
            for mode, name in FAMILIES:
                eng.set_fast_path(mode)
                got = host(eng.edges(d, ec))
                assert np.array_equal(got, want), (name, oi, ci, ks)
    eng.set_fast_path(True)


def test_element_larger_than_image(eng):
    import omni_b200
    masks = _masks(20, 30, 5)
    for oi, ci in ITERS:
        ec = omni_b200.EdgeConfig(ksize=3, morph_k=63, open_iters=oi, close_iters=ci)
        want = _want(masks, ec)
        for mode, name in FAMILIES:
            eng.set_fast_path(mode)
            assert np.array_equal(host(eng.edges(dev(masks), ec)), want), (name, oi, ci)
    eng.set_fast_path(True)


@pytest.mark.parametrize("oi,ci", [(40, 0), (0, 40), (33, 33)])
@pytest.mark.parametrize("mk", [3, 5])
def test_counts_past_32(eng, mk, oi, ci):
    import omni_b200
    masks = np.stack([blob_mask(150, 230, 7, 0.5, k=15), blob_mask(150, 230, 8, 0.3, k=21)])
    ec = omni_b200.EdgeConfig(ksize=3, morph_k=mk, open_iters=oi, close_iters=ci)
    want = _want(masks, ec)
    for mode, name in FAMILIES:
        eng.set_fast_path(mode)
        assert np.array_equal(host(eng.edges(dev(masks), ec)), want), name
    eng.set_fast_path(True)


@pytest.mark.parametrize("mk", [9, 16, 31])
def test_nonbinary_masks(eng, mk):
    """Hand-edited mask.png files with any u8 values take the generic byte kernel, now with per-row spans of any size."""
    import omni_b200
    masks = np.stack([smooth_u8(160, 250, 3), smooth_u8(160, 250, 4, k=11)])
    for oi, ci in ((1, 1), (2, 0), (0, 2)):
        ec = omni_b200.EdgeConfig(low=10, high=60, ksize=3, morph_k=mk, open_iters=oi, close_iters=ci)
        want = _want(masks, ec)
        for mode, name in FAMILIES:
            eng.set_fast_path(mode)
            assert np.array_equal(host(eng.edges(dev(masks), ec)), want), (name, oi, ci)
    eng.set_fast_path(True)


def test_fast_family_runs_the_bit_kernel(eng):
    """Binary masks at a size outside fk_morph go through the ELLIPSE bit-plane kernel, not the generic byte kernel."""
    import omni_b200
    masks = dev(_masks(300, 400, 11))
    eng.set_fast_path(True)
    ec = omni_b200.EdgeConfig(ksize=3, morph_k=9, open_iters=2, close_iters=1)
    eng.edges(masks, ec)
    torch.cuda.synchronize()
    eng.profile(True)
    eng.edges(masks, ec)
    prof = eng.profile_summary()
    eng.profile(False)
    assert prof.get("morph_ellipse_bits", (0, 0))[0] == 6 and "morph" not in prof, prof


ENTRY_EC = dict(ksize=3, morph_k=9, open_iters=2, close_iters=1)


@pytest.mark.parametrize("mode", [1, 3, 2, 0], ids=["fast", "fast_dense_pipeline", "fast_dense_edges", "generic"])
def test_entry_points_k9(eng, mode):
    """Every entry point at k=9, open 2, close 1: against the oracle and against its byte-plane twin."""
    import omni_b200
    ec = omni_b200.EdgeConfig(**ENTRY_EC)
    eng.set_fast_path(mode)
    try:
        # edges / host_edges
        masks = _masks(211, 389, 21)
        want = _want(masks, ec)
        got = host(eng.edges(dev(masks), ec))
        assert np.array_equal(got, want)
        assert np.array_equal(eng.host_edges(masks, ec), got)
        # color_edge (+ host_color_edge)
        K = 6
        img = synth(301, 517, 5, cell=16)
        ctr, lut = _centres(img, K)
        labels, m, e = eng.color_edge(dev(img), ctr, lut, ec, want_labels=True)
        m, e = host(m), host(e)
        assert np.array_equal(e, _want(m, ec))
        r = eng.host_color_edge(img, ctr, lut, ec)
        assert np.array_equal(r["masks"], m) and np.array_equal(r["edges"], e)
        # color_edge_packed, both bit orders
        for msb in (True, False):
            order = "big" if msb else "little"
            mb, eb = eng.color_edge_packed(dev(img), ctr, lut, ec, msb_first=msb)
            assert np.array_equal(host(mb), np.packbits(m > 0, axis=2, bitorder=order))
            assert np.array_equal(host(eb), np.packbits(e > 0, axis=2, bitorder=order))
        # color_edge_batch: 4 frames, K=8
        K = 8
        frames = np.stack([synth(190, 270, 40 + f, cell=16) for f in range(4)])
        ctr, lut = _centres(frames[0], K)
        bm, be = eng.color_edge_batch(dev(frames), ctr, lut, ec)
        bm, be = host(bm), host(be)
        for f in range(4):
            _l, m1, e1 = eng.color_edge(dev(frames[f]), ctr, lut, ec)
            assert np.array_equal(bm[f], host(m1)) and np.array_equal(be[f], host(e1)), f
            assert np.array_equal(be[f], _want(bm[f], ec)), f
    finally:
        eng.set_fast_path(True)


def test_host_packed_banded_size(eng):
    """host_color_edge_packed on one 1024 x 2048 frame (large enough for the banded path, which declines these parameters)."""
    import omni_b200
    ec = omni_b200.EdgeConfig(**ENTRY_EC)
    K = 8
    img = synth(1024, 2048, 9)
    ctr, lut = _centres(img, K)
    _l, m, e = eng.color_edge(dev(img), ctr, lut, ec)
    m, e = host(m), host(e)
    assert np.array_equal(e, _want(m, ec))
    r = eng.host_color_edge_packed(img, ctr, lut, ec)
    assert np.array_equal(r["mask_bits"], np.packbits(m > 0, axis=2))
    assert np.array_equal(r["edge_bits"], np.packbits(e > 0, axis=2))
    assert np.array_equal(r["counts"][:, 2], (e > 0).reshape(K, -1).sum(1))


@pytest.mark.parametrize("mode", [1, 0], ids=["fast", "generic"])
def test_strided_planes(eng, mode):
    """Planes that are views with row gaps: the result is right and nothing outside the view is written."""
    import omni_b200
    ec = omni_b200.EdgeConfig(ksize=3, morph_k=16, open_iters=1, close_iters=2)
    K, h, w = 3, 97, 301
    masks = np.stack([blob_mask(h, w, 60 + k, 0.4, k=7) for k in range(K)])
    want = _want(masks, ec)
    eng.set_fast_path(mode)
    try:
        big_in = torch.full((K, h, w + 45), 255, dtype=torch.uint8, device="cuda")
        big_in[:, :, 13:13 + w] = dev(masks)
        big_out = torch.full((K, h + 2, w + 51), 77, dtype=torch.uint8, device="cuda")
        view = big_out[:, 1:1 + h, 20:20 + w]
        eng.edges(big_in[:, :, 13:13 + w], ec, out=view)
        bo = host(big_out)
        assert np.array_equal(bo[:, 1:1 + h, 20:20 + w], want)
        bo[:, 1:1 + h, 20:20 + w] = 77
        assert (bo == 77).all()
        # host buffers: a view into a wider array
        hb = np.full((K, h, w + 29), 77, np.uint8)
        eng.host_edges(masks, ec, out=hb[:, :, 5:5 + w])
        assert np.array_equal(hb[:, :, 5:5 + w], want)
        hb[:, :, 5:5 + w] = 77
        assert (hb == 77).all()
    finally:
        eng.set_fast_path(True)


def test_4096_k16(eng):
    """BASELINE-sized planes: 4096^2, K=16, k=9, checked against the oracle on a few planes."""
    import omni_b200
    K = 16
    img = synth(4096, 4096, 0, cell=32)
    ctr, lut = _centres(img, K)
    masks = eng.color_edge(dev(img), ctr, lut, omni_b200.EdgeConfig())[1]
    ec = omni_b200.EdgeConfig(ksize=3, morph_k=9, open_iters=1, close_iters=1)
    got = eng.edges(masks, ec)
    m = host(masks)
    for k in (0, 7, 15):
        assert np.array_equal(host(got[k]), _want(m[k:k + 1], ec)[0]), k


def test_morph_k_bounds(eng):
    import omni_b200
    masks = _masks(40, 50, 3)
    with pytest.raises(omni_b200.OmniError, match="255"):
        eng.edges(dev(masks), omni_b200.EdgeConfig(morph_k=256))
    assert omni_b200.capi.OMNI_MAX_MORPH_K == 255
    ec = omni_b200.EdgeConfig(ksize=3, morph_k=255, open_iters=1, close_iters=1)
    assert np.array_equal(host(eng.edges(dev(masks), ec)), _want(masks, ec))


def _run_stage(script, cfg_path):
    env = dict(os.environ, CONFIG_PATH=cfg_path, PYTHONUNBUFFERED="1")
    r = subprocess.run([sys.executable, os.path.join(SCRIPTS, script)], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:]
    return r.stdout


def test_stages_02_03_k9(tmp_path):
    """config.json with edge_morph_kernel 9, open 2, close 1: stages 02 and 03 run as subprocesses, every edges.png is cv2's result
    for its mask.png, and stage 03 publishes the planes stage 02 parked instead of recomputing them."""
    rp = _rp()
    z, meta = load_pipe_case(PIPE_CASES[0])
    cfg = dict(meta["config"], edge_morph_kernel=9, edge_morph_open_iters=2, edge_morph_close_iters=1)
    names = meta["names"]
    out = tmp_path / "out"
    out.mkdir()
    cv2.imwrite(str(out / "resized.png"), z["resized"])
    cfg.update(input_image=str(tmp_path / "unused.png"), output_dir=str(out))
    cfg_path = out / "config.json"
    cfg_path.write_text(json.dumps(cfg))
    _run_stage("02_color_extract.py", str(cfg_path))
    assert (out / ".omni_b200_handoff.json").exists()
    parked = {n: (out / n / ".edges_b200.png").read_bytes() for n in names}
    log = _run_stage("03_edge_detect.py", str(cfg_path))
    assert not (out / ".omni_b200_handoff.json").exists()
    for n in names:
        m = cv2.imread(str(out / n / "mask.png"), cv2.IMREAD_GRAYSCALE)
        want = rp.edge_layer(m, cfg["edge_low_threshold"], cfg["edge_high_threshold"], cfg["edge_kernel_size"], 9, 2, 1)
        assert (out / n / "edges.png").read_bytes() == parked[n], n                  # published, not recomputed
        assert np.array_equal(cv2.imread(str(out / n / "edges.png"), cv2.IMREAD_GRAYSCALE), want), n
        assert f"Edges extracted: {n} | nz={int(np.count_nonzero(want))}" in log
