"""PNG files encoded on the GPU (omni_png_encode / omni_host_png_encode, csrc/png_encode.cu).

Every file is decoded by cv2 (libpng) and must give back exactly the source pixels; its chunks are walked with every CRC,
the IHDR fields and the chunk order checked; its IDAT stream must inflate to its end with nothing left over (which also
checks the Adler-32).  Then: the Huffman length limit, strides and batches, device form = host form, determinism across
calls / streams / contexts, the argument errors, the sizes against the encoders the stages used before, and the files the
stage scripts write."""
import json
import os
import struct
import zlib

import cv2
import numpy as np
import pytest

from helpers import synth

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _omni():
    import omni_b200
    return omni_b200


GRAY1, BGR8 = 0, 1


@pytest.fixture(scope="module")
def eng():
    e = _omni().Engine(0)
    yield e
    e.close()


@pytest.fixture
def fresh():
    e = _omni().Engine(0)
    yield e
    e.close()


def seg_rows(w, fmt):
    """Rows per segment, as include/omni_b200.h states the rule."""
    row = (w + 7) // 8 if fmt == GRAY1 else 3 * w
    return max(1, min(256, 61440 // (row + 1)))


def chunks(png: bytes):
    """[(type, data)] after checking the signature, every CRC and the order IHDR, IDAT..., IEND."""
    assert png[:8] == b"\x89PNG\r\n\x1a\n"
    out, o = [], 8
    while o < len(png):
        n, = struct.unpack(">I", png[o:o + 4])
        t, d = png[o + 4:o + 8], png[o + 8:o + 8 + n]
        crc, = struct.unpack(">I", png[o + 8 + n:o + 12 + n])
        assert crc == zlib.crc32(t + d) & 0xFFFFFFFF, f"bad CRC in {t} at {o}"
        out.append((t, d))
        o += 12 + n
    assert o == len(png)
    types = [t for t, _ in out]
    assert types[0] == b"IHDR" and types[-1] == b"IEND" and set(types[1:-1]) == {b"IDAT"}, types
    return out


def check_file(png: bytes, src: np.ndarray, fmt: int, w: int):
    """src: packed rows [H, RB] (GRAY1) or BGR [H, W, 3]."""
    ch = chunks(png)
    h = src.shape[0]
    assert ch[0][1] == struct.pack(">IIBBBBB", w, h, 1 if fmt == GRAY1 else 8, 0 if fmt == GRAY1 else 2, 0, 0, 0)
    z = zlib.decompressobj()
    raw = z.decompress(b"".join(d for t, d in ch if t == b"IDAT"))
    assert z.eof and not z.unused_data and not z.unconsumed_tail
    rowlen = ((w + 7) // 8 if fmt == GRAY1 else 3 * w) + 1
    assert len(raw) == h * rowlen
    dec = cv2.imdecode(np.frombuffer(png, np.uint8), cv2.IMREAD_UNCHANGED)
    if fmt == GRAY1:
        want = np.unpackbits(src, axis=1)[:, :w] * np.uint8(255)
        assert dec.shape == (h, w) and np.array_equal(dec, want)
    else:
        assert dec.shape == src.shape and np.array_equal(dec, src)


def enc_check(eng, a, fmt, w=None, host=True):
    files = eng.host_png_encode(a, fmt, w) if host else eng.png_encode(torch.from_numpy(np.ascontiguousarray(a)).cuda(), fmt, w)
    imgs = a if a.ndim == (3 if fmt == GRAY1 else 4) else a[None]
    assert len(files) == len(imgs)
    for f, im in zip(files, imgs):
        iw = im.shape[1] if fmt == BGR8 else (w if w is not None else 8 * im.shape[1])
        check_file(f, np.ascontiguousarray(im), fmt, iw)
        assert len(f) <= eng._L.omni_png_bound(im.shape[0], iw, fmt)
    return files


def bits(h, w, seed, kind="noise"):
    rb = (w + 7) // 8
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, rb), dtype=np.uint8)
    if kind == "zeros":
        return np.zeros((h, rb), np.uint8)
    if kind == "ones":
        return np.full((h, rb), 255, np.uint8)
    if kind == "alt":
        return np.tile(np.array([0x55, 0xAA], np.uint8), (h, rb + 1))[:, :rb].copy()
    m = (cv2.GaussianBlur(rng.integers(0, 256, (h, w), dtype=np.uint8), (0, 0), 3) > 128)
    return np.packbits(m, axis=1)


def bgr(h, w, seed, kind="synth"):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "zeros":
        return np.zeros((h, w, 3), np.uint8)
    if kind == "ones":
        return np.full((h, w, 3), 255, np.uint8)
    if kind == "alt":
        return np.tile(np.array([0, 255], np.uint8), (h * w * 3 + 1))[:h * w * 3].reshape(h, w, 3).copy()
    return synth(h, w, seed, cell=16) if min(h, w) >= 16 else rng.integers(0, 256, (h, w, 3), dtype=np.uint8)


# ---- shapes and contents ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w", list(range(1, 18)) + [4095, 4096, 4097])
@pytest.mark.parametrize("kind", ["noise", "zeros", "ones", "alt", "blobs"])
def test_gray1_widths(eng, w, kind):
    h = 37 if w < 4000 else 300
    enc_check(eng, bits(h, w, w, kind), GRAY1, w)


@pytest.mark.parametrize("shape", [(1, 1), (1, 97), (97, 1), (67, 93), (1080, 1920)])
@pytest.mark.parametrize("kind", ["noise", "zeros", "ones", "alt", "synth"])
def test_bgr8_shapes(eng, shape, kind):
    enc_check(eng, bgr(*shape, seed=shape[0] + shape[1], kind=kind), BGR8)


@pytest.mark.parametrize("shape", [(1, 1), (1, 64), (64, 1), (67, 93), (1080, 1920)])
def test_gray1_shapes(eng, shape):
    h, w = shape
    enc_check(eng, bits(h, w, 3, "blobs" if min(h, w) > 8 else "noise"), GRAY1, w)


def test_4096_square(eng):
    enc_check(eng, bgr(4096, 4096, 1), BGR8)
    enc_check(eng, bits(4096, 4096, 2, "blobs"), GRAY1, 4096)


@pytest.mark.parametrize("fmt,w", [(GRAY1, 1920), (GRAY1, 100), (BGR8, 1920), (BGR8, 93)])
@pytest.mark.parametrize("dh", [-1, 0, 1])
def test_heights_around_a_segment(eng, fmt, w, dh):
    h = seg_rows(w, fmt) + dh
    a = bits(h, w, h, "blobs") if fmt == GRAY1 else bgr(h, w, h)
    enc_check(eng, a, fmt, w if fmt == GRAY1 else None)
    enc_check(eng, np.concatenate([a, a]), fmt, w if fmt == GRAY1 else None)     # two segments and a bit


def test_one_row_segments(eng):
    w = 10240                                   # 3 * w + 1 > 61440 / 2: one row per segment
    assert seg_rows(w, BGR8) == 1
    enc_check(eng, bgr(5, w, 0), BGR8)
    enc_check(eng, bgr(3, w, 0, "zeros"), BGR8)
    assert seg_rows(20479, BGR8) == 1
    enc_check(eng, bgr(2, 20479, 0, "noise"), BGR8)


def test_long_runs_cross_rows_and_segments(eng):
    # runs far longer than 258 bytes through scanline and segment boundaries, with short interruptions
    h, w = 3 * seg_rows(4096, GRAY1) + 5, 4096
    a = np.zeros((h, 512), np.uint8)
    a[5, 100] = 1
    a[h // 2:, :] = 255
    a[h // 2 + 3, 7] = 0x0F
    enc_check(eng, a, GRAY1, w)
    b = np.zeros((300, 700, 3), np.uint8)
    b[150:] = 255
    b[100, 3] = (1, 2, 3)
    enc_check(eng, b, BGR8)
    for m in (1, 2, 3, 4, 258, 259, 260, 261, 262, 516, 517):     # run lengths around the match limits
        r = np.full((1, 2000), 7, np.uint8)
        r[0, 1 + m:] = 9
        enc_check(eng, r, GRAY1, 16000)


def test_fibonacci_needs_the_length_limit(eng):
    """Byte frequencies 1, 1, 2, 3, 5, ... with no value twice in a row: every byte is a literal and an unlimited Huffman
    code would be deeper than 15 bits."""
    fib = [1, 1]
    while sum(fib) + fib[-1] + fib[-2] < 30000:
        fib.append(fib[-1] + fib[-2])
    assert len(fib) > 17
    counts = {v: f for v, f in enumerate(fib)}
    seq = []
    # greedy interleave so that no value repeats back to back: always take the most frequent value that is not the last one
    left = dict(counts)
    last = None
    while left:
        cand = sorted(left.items(), key=lambda kv: (-kv[1], kv[0]))
        v = cand[0][0] if cand[0][0] != last else (cand[1][0] if len(cand) > 1 else None)
        if v is None:
            break
        seq.append(v)
        left[v] -= 1
        if left[v] == 0:
            del left[v]
        last = v
    data = np.array(seq, np.uint8) + 1           # values 1..: never equal to the filter byte 0 in front of each row
    rb = 240
    h = len(data) // rb
    a = data[:h * rb].reshape(h, rb)
    assert (a[:, 1:] != a[:, :-1]).all()
    f = enc_check(eng, a, GRAY1, 8 * rb)[0]
    assert len(f) < a.size                       # compressed (not stored): the dynamic code was built and limited


# ---- strides, batches, device = host -----------------------------------------------------------------------------------
def test_strided_and_sliced(eng):
    big = bgr(300, 400, 5)
    view = big[10:250:2, 30:330]                 # row stride 2 * pitch, column offset
    f = enc_check(eng, view, BGR8)[0]
    assert f == eng.host_png_encode(np.ascontiguousarray(view), BGR8)[0]
    pb = bits(200, 800, 6, "blobs")
    v2 = pb[:, 3:53]                             # packed rows inside wider rows
    g = enc_check(eng, v2, GRAY1, 400)[0]
    assert g == eng.host_png_encode(np.ascontiguousarray(v2), GRAY1, 400)[0]
    d = torch.from_numpy(big).cuda()[10:250:2, 30:330]
    assert eng.png_encode(d, BGR8)[0] == f


def test_batches(eng):
    planes = np.stack([bits(500, 1000, s, k) for s, k in enumerate(["blobs", "zeros", "noise", "ones", "alt", "blobs"])])
    files = enc_check(eng, planes, GRAY1, 1000)
    for p, f in zip(planes, files):
        assert eng.host_png_encode(p, GRAY1, 1000)[0] == f
    strided = planes[::2]
    assert eng.host_png_encode(strided, GRAY1, 1000) == files[::2]
    imgs = np.stack([bgr(120, 77, s) for s in range(3)])
    enc_check(eng, imgs, BGR8)
    d = torch.from_numpy(planes).cuda()
    assert eng.png_encode(d, GRAY1, 1000) == files
    assert eng.png_encode(d[1::2], GRAY1, 1000) == files[1::2]


def test_device_equals_host(eng):
    for a, fmt, w in [(bgr(1080, 1920, 9), BGR8, None), (bits(1080, 1920, 9, "blobs"), GRAY1, 1920), (bgr(67, 93, 2, "noise"), BGR8, None)]:
        assert enc_check(eng, a, fmt, w, host=False) == eng.host_png_encode(a, fmt, w)


# ---- determinism ---------------------------------------------------------------------------------------------------
def test_repeatable_across_calls_streams_and_contexts(eng, fresh):
    a = np.stack([bits(700, 1500, s, "blobs") for s in range(4)])
    b = bgr(500, 600, 3)
    ref_a, ref_b = eng.host_png_encode(a, GRAY1, 1500), eng.host_png_encode(b, BGR8)
    for _ in range(3):
        assert eng.host_png_encode(a, GRAY1, 1500) == ref_a
        assert eng.host_png_encode(b, BGR8) == ref_b
    eng.host_png_encode(bgr(2000, 3000, 1), BGR8)         # a larger call grows the scratch in between
    assert eng.host_png_encode(a, GRAY1, 1500) == ref_a
    assert fresh.host_png_encode(b, BGR8) == ref_b
    assert fresh.host_png_encode(a, GRAY1, 1500) == ref_a
    da = torch.from_numpy(a).cuda()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(s1):
        r1 = eng.png_encode(da, GRAY1, 1500)
    with torch.cuda.stream(s2):
        r2 = eng.png_encode(da, GRAY1, 1500)
    assert r1 == ref_a and r2 == ref_a


def test_interleaved_with_fused_calls(fresh):
    """Encoder calls between fused colour/edge calls on one context change neither side's results."""
    import omni_b200
    img = synth(720, 1280, 4, cell=16)
    ctr = np.array([[40, 128, 128], [110, 140, 120], [160, 120, 150], [220, 128, 128]], np.float32)
    lut = np.arange(4, dtype=np.uint8)
    ec = omni_b200.EdgeConfig()
    ref_fused = fresh.host_color_edge_packed(img, ctr, lut, ec, msb_first=True)
    ref_files = omni_b200.Engine(0).host_png_encode(ref_fused["mask_bits"], GRAY1, 1280)
    files = fresh.host_png_encode(ref_fused["mask_bits"], GRAY1, 1280)
    again = fresh.host_color_edge_packed(img, ctr, lut, ec, msb_first=True)
    files2 = fresh.host_png_encode(again["edge_bits"], GRAY1, 1280)
    third = fresh.host_color_edge_packed(img, ctr, lut, ec, msb_first=True)
    assert files == ref_files
    for k in ("mask_bits", "edge_bits", "counts"):
        assert np.array_equal(again[k], ref_fused[k]) and np.array_equal(third[k], ref_fused[k])
    assert files2 == omni_b200.Engine(0).host_png_encode(ref_fused["edge_bits"], GRAY1, 1280)
    d = fresh.png_encode(torch.from_numpy(img).cuda(), BGR8)
    assert d == fresh.host_png_encode(img, BGR8)


# ---- arguments -----------------------------------------------------------------------------------------------------
def test_invalid_arguments(eng):
    import ctypes as C
    L, h = eng._L, eng._h
    d = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
    out = torch.zeros(1 << 22, dtype=torch.uint8, device="cuda")
    sizes = np.zeros(4, np.int64)
    sp = sizes.ctypes.data_as(C.POINTER(C.c_int64))
    big = 1 << 22

    def call(n=1, stride=0, hh=4, w=8, pitch=8, fmt=GRAY1, cap=big):
        rc = L.omni_png_encode(h, d.data_ptr(), n, stride, hh, w, pitch, fmt, out.data_ptr(), cap, sp, None)
        return rc, L.omni_last_error_string().decode()

    assert call()[0] == 0
    for kw, text in [(dict(fmt=7), "unknown format 7"), (dict(hh=0), "at least 1"), (dict(w=0), "at least 1"),
                     (dict(pitch=0), "shorter than a row"), (dict(fmt=BGR8, w=8, pitch=23), "shorter than a row"),
                     (dict(cap=10), "omni_png_bound"), (dict(n=2, cap=L.omni_png_bound(4, 8, GRAY1) * 2 - 1), "omni_png_bound"),
                     (dict(fmt=BGR8, w=20480, pitch=3 * 20480), "OMNI_PNG_MAX_SCANLINE = 61440"),
                     (dict(fmt=GRAY1, w=491513, pitch=61440), "OMNI_PNG_MAX_SCANLINE = 61440"),
                     (dict(hh=(1 << 24) + 1), "OMNI_PNG_MAX_ROWS"), (dict(n=0), "at least 1")]:
        rc, msg = call(**kw)
        assert rc == -1, (kw, rc)
        assert text in msg, (kw, msg)
    assert L.omni_png_bound(0, 5, GRAY1) == 0 and L.omni_png_bound(5, 5, 3) == 0 and L.omni_png_bound(5, 20480, BGR8) == 0
    assert L.omni_png_bound(5, 20479, BGR8) > 0
    with pytest.raises(_omni().OmniError, match="unknown format"):
        eng.host_png_encode(np.zeros((4, 4), np.uint8), 5)


# ---- sizes against the encoders the stages used --------------------------------------------------------------------
def _stage_planes(eng, h, w, K, seed):
    from omni_b200 import stages, synth as osynth
    img = osynth.synth(h, w, seed)
    centers = stages.kmeans_lab_centers(img, K)
    order, lut = stages.darkness_lut(centers)
    r = eng.host_color_edge_packed(img, centers, lut.astype(np.uint8), _omni().EdgeConfig(), msb_first=True)
    return img, r["mask_bits"], r["edge_bits"]


@pytest.mark.parametrize("h,w,K", [(4096, 4096, 8), (4096, 4096, 16), (1080, 1920, 8)])
def test_sizes(eng, h, w, K):
    from omni_b200 import png1
    img, mb, eb = _stage_planes(eng, h, w, K, seed=K)
    for planes in (mb, eb):
        new = eng.host_png_encode(planes, GRAY1, w)
        old = [png1.encode_png1(p, w) for p in planes]
        for f, p in zip(new[:2], planes[:2]):
            check_file(f, p, GRAY1, w)
        assert sum(map(len, new)) <= sum(map(len, old)), (sum(map(len, new)), sum(map(len, old)))
    f = eng.host_png_encode(img, BGR8)[0]
    check_file(f, img, BGR8, w)
    assert len(f) <= 1.02 * len(cv2.imencode(".png", img)[1])
    rng = np.random.default_rng(7)
    stack = np.unpackbits(eb, axis=2)[:, :, :w] * np.uint8(255)
    canvas = eng.host_edges_composite(stack, [tuple(int(v) for v in rng.integers(0, 256, 3)) for _ in range(K)])
    c = eng.host_png_encode(canvas, BGR8)[0]
    check_file(c, canvas, BGR8, w)
    assert len(c) <= len(cv2.imencode(".png", canvas)[1])


# ---- the files the stage scripts write ---------------------------------------------------------------------------------
def _same_as_encoder(eng, out, names):
    for n in names:
        for f in ("mask.png", "edges.png"):
            p = os.path.join(out, n, f)
            m = cv2.imread(p, cv2.IMREAD_GRAYSCALE)
            assert open(p, "rb").read() == eng.host_png_encode(np.packbits(m > 0, axis=1), GRAY1, m.shape[1])[0], p
    for f in ("resized.png", "edges_composite.png"):
        p = os.path.join(out, f)
        assert open(p, "rb").read() == eng.host_png_encode(cv2.imread(p, cv2.IMREAD_COLOR), BGR8)[0], p


@pytest.mark.parametrize("front_half", [False, True])
def test_stage_files_are_the_encoder_output(eng, tmp_path, front_half):
    import subprocess
    import sys
    scripts = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "omnirevolve-image-processor_b200",
                           "image_processor")
    src = tmp_path / "input.png"
    cv2.imwrite(str(src), synth(700, 900, 3))
    names = ["layer_dark", "layer_mid", "layer_skin", "layer_light"]
    out = tmp_path / "out"
    out.mkdir()
    cfg = {"input_image": str(src), "output_dir": str(out), "max_dimension": 800, "color_names": names,
           "colors": [[0, 0, 0], [255, 0, 0], [0, 255, 0], [0, 0, 255]]}
    (out / "config.json").write_text(json.dumps(cfg))
    env = dict(os.environ, CONFIG_PATH=str(out / "config.json"))
    for s in (["front_half.py"] if front_half else ["01_resize.py", "02_color_extract.py", "03_edge_detect.py"]):
        r = subprocess.run([sys.executable, os.path.join(scripts, s)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                           text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-3000:]
    _same_as_encoder(eng, str(out), names)
    # stage 03 run alone (no hand-off): detect_all_edges / save_edges_composite write the files
    for n in names:
        os.remove(out / n / "edges.png")
    os.remove(out / "edges_composite.png")
    r = subprocess.run([sys.executable, os.path.join(scripts, "03_edge_detect.py")], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:]
    _same_as_encoder(eng, str(out), names)
