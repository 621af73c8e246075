"""Packed edge planes -> centrelines in one call (omni_centerlines_packed / omni_host_centerlines_packed, csrc/trace.cu): every
plane's result equals the composition of the existing calls -- omni_thin_zhangsuen_packed, unpacking to {0,255} bytes,
omni_trace_centerlines (at most 32 planes each) -- for batches that span several chunks of planes, odd geometries, both bit
orders, padded pitches and plane strides; the host walk, the call order, contours.trace_frames and the argument checks."""
import contextlib
import ctypes as C
import io
import os
import subprocess
import sys

import cv2
import numpy as np
import pytest

from conftest import ROOT
from helpers import synth

pytestmark = pytest.mark.gpu

H, W, K = 1080, 1920, 8


@pytest.fixture(scope="module")
def eng():
    import omni_b200
    return omni_b200.get_engine()


def _unpack(bits, w, msb):
    return np.unpackbits(bits, axis=-1, bitorder="big" if msb else "little")[..., :w] * np.uint8(255)


def _pack(planes, msb):
    return np.packbits(planes > 0, axis=-1, bitorder="big" if msb else "little")


def _compose(eng, bits, w, max_iter=120, msb=True):
    """The existing calls, at most 32 planes each: packed thinning, unpacking on the host, omni_trace_centerlines."""
    import torch
    d = torch.from_numpy(np.ascontiguousarray(bits)).cuda()
    out = []
    for g in range(0, d.shape[0], 32):
        thin = eng.thin_zhangsuen_packed(d[g:g + 32], w, max_iter, msb_first=msb)
        out += eng.trace_centerlines(torch.from_numpy(_unpack(thin.cpu().numpy(), w, msb)).cuda())
    return out


def _same(a, b):
    assert a.total_fg == b.total_fg
    assert a.stats.shape == b.stats.shape and np.array_equal(a.stats, b.stats)
    assert np.array_equal(a.polylines, b.polylines) and len(a.paths) == len(b.paths)
    assert [len(p) for p in a.paths] == [len(p) for p in b.paths]
    if a.paths:
        assert all(p.dtype == np.int32 and p.shape[1:] == (1, 2) for p in a.paths)
        assert np.array_equal(np.concatenate(a.paths), np.concatenate(b.paths))


def _same_all(xs, ys):
    assert len(xs) == len(ys)
    for x, y in zip(xs, ys):
        _same(x, y)


def _padded(bits, dev):
    """The planes as a view with pitch > ceil(w/8), plane stride > pitch * h and an offset start."""
    P, h, rb = bits.shape
    if dev:
        import torch
        buf = torch.zeros((P + 2, h + 3, rb + 5), dtype=torch.uint8, device="cuda")
        buf[1:P + 1, 2:h + 2, 3:rb + 3] = torch.from_numpy(np.ascontiguousarray(bits)).cuda()
    else:
        buf = np.zeros((P + 2, h + 3, rb + 5), np.uint8)
        buf[1:P + 1, 2:h + 2, 3:rb + 3] = bits
    return buf[1:P + 1, 2:h + 2, 3:rb + 3]


@pytest.fixture(scope="module")
def frames_1080(eng):
    """25 configs[3]-style 1080p frames, K = 8: 200 packed edge planes (MSB first) and the composition result of every plane."""
    from omni_b200 import EdgeConfig
    n = 25
    imgs = np.stack([synth(H, W, s) for s in range(n)])
    ctr = np.array([[25 + 30 * i, 100 + 8 * i, 160 - 7 * i] for i in range(K)], np.float32)
    bits = eng.host_color_edge_packed(imgs, ctr, np.arange(K, dtype=np.uint8), EdgeConfig(), want_counts=False)["edge_bits"]
    return bits, _compose(eng, bits, W)


@pytest.mark.parametrize("P", [8, 32, 33, 64, 200])
def test_centerlines_packed_1080p_equals_composition(eng, frames_1080, P):
    """200 planes at 1080p are 4 chunks of at most 64 planes."""
    import torch
    bits, want = frames_1080
    got = eng.centerlines_packed(torch.from_numpy(bits[:P]).cuda(), W)
    _same_all(got, want[:P])
    assert sum(len(r.paths) for r in got) > 0


def test_centerlines_packed_1080p_lsb_first_padded_host(eng, frames_1080):
    bits, want = frames_1080
    lsb = np.packbits(np.unpackbits(bits[:40], axis=2, bitorder="big"), axis=2, bitorder="little")
    _same_all(eng.host_centerlines_packed(_padded(lsb, False), W, msb_first=False), want[:40])


def _noise_planes(P, h, w, seed):
    """Thick noise (junction-rich, wandering cycles), sparse noise, empty planes, a few lines: 40 planes cross a thinning group."""
    rng = np.random.default_rng(seed)
    p = np.zeros((P, h, w), np.uint8)
    for i in range(P):
        kind = i % 4
        if kind == 0:
            p[i] = (rng.random((h, w)) < 0.35) * 255
        elif kind == 1:
            p[i] = (rng.random((h, w)) < 0.08) * 255
        elif kind == 2:
            cv2.line(p[i], (0, int(rng.integers(0, h))), (w - 1, int(rng.integers(0, h))), 255, 1 + i % 3)
    return p


@pytest.mark.parametrize("shape", [(67, 93), (40, 1), (33, 7), (50, 9), (45, 129)])
@pytest.mark.parametrize("msb", [True, False])
def test_centerlines_packed_geometries_and_bit_orders(eng, shape, msb):
    h, w = shape
    planes = _noise_planes(40, h, w, h * 1000 + w)
    bits = _pack(planes, msb)
    want = _compose(eng, bits, w, msb=msb)
    _same_all(eng.centerlines_packed(_padded(bits, True), w, msb_first=msb), want)
    _same_all(eng.host_centerlines_packed(_padded(bits, False), w, msb_first=msb), want)
    for it in (0, 3):                                            # max_iter passes through to the thinning
        _same_all(eng.host_centerlines_packed(bits, w, max_iter=it, msb_first=msb), _compose(eng, bits, w, it, msb))


def _maps(sk):
    S = (sk > 0).astype(np.uint8)
    k = np.ones((3, 3), np.uint8)
    k[1, 1] = 0
    deg = cv2.filter2D(S, cv2.CV_8U, k, borderType=cv2.BORDER_CONSTANT)
    return deg, (S == 1) & (deg == 1), (S == 1) & (deg >= 3)


def test_centerlines_packed_equals_host_walk(eng):
    from omni_b200 import contours
    planes = _noise_planes(6, 61, 83, 5)
    res = eng.host_centerlines_packed(_pack(planes, True), 83)
    sks = eng.host_thin_zhangsuen(planes)[0]
    for r, sk in zip(res, sks):
        with contextlib.redirect_stdout(io.StringIO()):
            paths = contours._trace_host(sk, "L", _maps(sk))
        assert len(paths) == len(r.paths) and all(np.array_equal(a, b) for a, b in zip(paths, r.paths))
        num, _lab, st, _c = cv2.connectedComponentsWithStats((sk > 0).astype(np.uint8), connectivity=8)
        assert np.array_equal(r.stats, st[1:]) and r.total_fg == int((sk > 0).sum())


def test_centerlines_packed_mixed_content_across_chunks(eng):
    """1080p planes, 4 chunks (64, 64, 64, 8): components larger than the shared-memory window (a frame on the border with
    paths and a loop attached) in the first, a middle and the last chunk, empty planes, a single-pixel plane, small content."""
    P = 200
    planes = np.zeros((P, H, W), np.uint8)
    for i in (0, 100, 199):
        a = planes[i]
        a[0, :] = a[-1, :] = a[:, 0] = a[:, -1] = 255
        for j in range(6):
            cv2.line(a, (0, 100 + 150 * j), (300 + 200 * j, 200 + 120 * j), 255, 1)
        cv2.circle(a, (1400, 500), 200 + i, 255, 1)
        cv2.line(a, (1200, 500), (900, 500), 255, 1)
    planes[63, 500, 700] = 255                                   # a single pixel, last plane of the first chunk
    planes[64, 0, 0] = 255                                       # a single pixel in a corner, first plane of the second chunk
    for i in (5, 70, 150):
        cv2.circle(planes[i], (300 + i, 400), 30, 255, 1)
        cv2.rectangle(planes[i], (1000, 100), (1100, 160), 255, 3)
    bits = _pack(planes, True)
    got = eng.host_centerlines_packed(bits, W)
    _same_all(got, _compose(eng, bits, W))
    st = [r.stats for r in got]
    assert all(((s[:, 2] + 2) * (s[:, 3] + 2) > 200 * 1024).any() for s in (st[0], st[100], st[199]))
    assert got[63].total_fg == 1 and got[63].paths == [] and got[63].stats.tolist() == [[700, 500, 1, 1, 1]]
    assert all(got[i].total_fg == 0 and got[i].paths == [] and got[i].stats.shape == (0, 5) for i in (1, 62, 65, 128, 198))


def test_centerlines_packed_all_empty(eng):
    import torch
    for P, h, w in ((130, H, W), (3, 5, 7)):                     # several chunks / one chunk, nothing in any plane
        res = eng.centerlines_packed(torch.zeros((P, h, (w + 7) // 8), dtype=torch.uint8, device="cuda"), w)
        assert len(res) == P and all(r.paths == [] and r.total_fg == 0 and r.stats.shape == (0, 5) for r in res)


def test_centerlines_packed_device_and_host_forms_agree(eng, frames_1080):
    import torch
    bits = frames_1080[0][64:100]
    dev = eng.centerlines_packed(_padded(bits, True), W)
    host = eng.host_centerlines_packed(_padded(bits, False), W)
    _same_all(dev, host)
    _same_all(dev, frames_1080[1][64:100])
    _same_all(eng.centerlines_packed(torch.from_numpy(bits).cuda(), W), host)


def test_call_order_with_trace_centerlines(eng, frames_1080):
    """A trace before and after the new call gives the same result; omni_trace_results returns the latest call's output."""
    import torch
    bits, want = frames_1080
    sk = _unpack(eng.thin_zhangsuen_packed(torch.from_numpy(bits[:8]).cuda(), W).cpu().numpy(), W, True)
    before = eng.host_trace_centerlines(sk)
    batch = eng.host_centerlines_packed(bits[:150], W)
    after = eng.host_trace_centerlines(sk)
    _same_all(before, after)
    _same_all(before, want[:8])
    _same_all(batch, want[:150])
    small = eng.host_centerlines_packed(bits[8:12], W)           # a smaller result after a larger one
    _same_all(small, want[8:12])
    info = np.array([[r.total_fg, len(r.stats), len(r.paths), sum(len(p) for p in r.paths)] for r in small], np.int64)
    assert np.array_equal(info, np.array([[w.total_fg, len(w.stats), len(w.paths), sum(len(p) for p in w.paths)]
                                          for w in want[8:12]], np.int64))
    _same_all(eng._trace_results(info), small)


def test_trace_centerlines_still_rejects_more_than_32_planes(eng):
    import torch
    import omni_b200
    with pytest.raises(omni_b200.OmniError):
        eng.trace_centerlines(torch.zeros((33, 8, 8), dtype=torch.uint8, device="cuda"))


def test_trace_frames_equals_per_frame_trace_centerlines(eng):
    from omni_b200 import EdgeConfig, contours
    n, k, h, w = 3, 4, 240, 333
    imgs = np.stack([synth(h, w, 50 + s) for s in range(n)])
    ctr = np.array([[40, 128, 128], [110, 140, 120], [160, 120, 150], [220, 128, 128]], np.float32)
    bits = eng.host_color_edge_packed(imgs, ctr, np.arange(k, dtype=np.uint8), EdgeConfig())["edge_bits"]
    with contextlib.redirect_stdout(io.StringIO()) as log:
        got = contours.trace_frames(bits, w, k)
    assert log.getvalue() == ""
    sks = eng.host_thin_zhangsuen(_unpack(bits, w, True))[0]
    assert len(got) == n and all(len(f) == k for f in got)
    with contextlib.redirect_stdout(io.StringIO()):
        for f in range(n):
            for j in range(k):
                want = contours.trace_centerlines(sks[f * k + j], f"f{f}l{j}")
                assert len(got[f][j]) == len(want) and all(np.array_equal(a, b) for a, b in zip(got[f][j], want))
    assert sum(len(p) for f in got for p in f) > 0
    with pytest.raises(ValueError):
        contours.trace_frames(bits[:5], w, k)


def test_argument_errors_leave_ctx_usable(eng):
    import omni_b200
    from omni_b200 import capi
    L = capi.lib()
    planes = _noise_planes(3, 20, 30, 1)
    bits = np.ascontiguousarray(_pack(planes, True))
    ps, pitch = bits.strides[0], bits.strides[1]
    want = eng.host_centerlines_packed(bits, 30)
    info = np.zeros((3, 4), np.int64)
    ip = info.ctypes.data_as(C.POINTER(C.c_int64))
    d = bits.ctypes.data
    bad = [
        (None, 3, 20, 30, ps, pitch, 1, 120),                    # null planes
        (d, 0, 20, 30, ps, pitch, 1, 120),                       # no planes
        (d, 3, 0, 30, ps, pitch, 1, 120),
        (d, 3, 20, 0, ps, pitch, 1, 120),
        (d, 3, 20, 30, ps, 3, 1, 120),                           # pitch < ceil(w / 8)
        (d, 3, 20, 30, pitch * 20 - 1, pitch, 1, 120),           # plane stride < pitch * h
        (d, 3, 20, 30, ps, pitch, 2, 120),                       # bit order
        (d, 3, 20, 30, ps, pitch, 1, -1),                        # max_iter
        (d, 3, 20, 30, ps, pitch, 1, 100001),
    ]
    for args in bad:
        rc = L.omni_host_centerlines_packed(eng._h, *args, ip)
        assert rc == -1, args
        assert b"omni_host_centerlines_packed" in L.omni_last_error_string()
        with pytest.raises(omni_b200.OmniError):
            capi.check(rc)
    rc = L.omni_centerlines_packed(eng._h, None, 3, 20, 30, ps, pitch, 1, 120, ip, None)
    assert rc == -1 and b"omni_centerlines_packed" in L.omni_last_error_string()
    with pytest.raises(ValueError):
        eng.host_centerlines_packed(bits, 30 * 8)                # rows too short for w
    _same_all(eng.host_centerlines_packed(bits, 30), want)


def test_host_form_does_not_import_torch():
    pkg = os.path.join(ROOT, "omnirevolve-image-processor_b200")
    code = ("import sys; sys.path.insert(0, %r); import numpy as np; import omni_b200; from omni_b200 import contours\n"
            "p = np.zeros((9, 40, 50), np.uint8); p[:, 5, 3:47] = 255; p[:, 9:30, 20] = 255\n"
            "bits = np.packbits(p > 0, axis=-1)\n"
            "res = omni_b200.get_engine().host_centerlines_packed(bits, 50)\n"
            "fr = contours.trace_frames(bits, 50, 3)\n"
            "n = len(res[0].paths)\n"
            "assert n > 0 and all(len(r.paths) == n for r in res) and len(fr) == 3 and all(len(f[1]) == n for f in fr)\n"
            "assert 'torch' not in sys.modules, 'torch imported'; print('NO_TORCH_OK')" % pkg)
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=300)
    assert r.returncode == 0 and "NO_TORCH_OK" in r.stdout, r.stdout[-2000:]
