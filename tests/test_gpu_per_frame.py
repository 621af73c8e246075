"""Frame batches in which every frame has its own colour centres.

- omni_kmeans_lab_batch: frame f's centres and compactness are bit-identical to omni_kmeans_lab on that frame alone.
- omni_color_edge_packed_frames / omni_host_color_edge_packed_frames: frame f's mask / edge bits and counts equal the shared-centre
  omni_color_edge_packed on that frame with centers[f] and lut[f], in every kernel family, both bit orders and the stage-03 variants.
- The candidate-table cache and the call order: per-frame and shared-centre calls on one context give what fresh contexts give.
Needs a B200: `-m gpu`."""
import ctypes as C

import numpy as np
import pytest

from helpers import synth, uniform_img

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

FAMILIES = (1, 3, 2, 0)          # label-domain pipeline (default), dense first generation, dense edges + Lab cells, generic


def _omni():
    import omni_b200
    return omni_b200


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


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


def frame(h, w, seed, kind="synth"):
    if kind == "flat":
        return np.full((h, w, 3), (seed * 37) % 256, np.uint8)
    if kind == "noise" or min(h, w) < 16:
        return uniform_img(h, w, seed)
    return synth(h, w, seed, cell=16)


def frames_of(n, h, w, seed, kinds=("synth",)):
    return np.stack([frame(h, w, seed + i, kinds[i % len(kinds)]) for i in range(n)])


def centres_of(img, K, seed):
    """K Lab centres near colours of the image (layers are populated), with fractional parts, and a darkness-style LUT."""
    from oracle import cmodel
    lab = cmodel.bgr2lab(img).reshape(-1, 3).astype(np.float32)
    rng = np.random.default_rng(seed)
    ctr = (lab[rng.integers(0, lab.shape[0], K)] + rng.uniform(-4, 4, (K, 3))).astype(np.float32)
    lut = np.zeros(K, np.uint8)
    lut[np.argsort(ctr[:, 0], kind="stable")] = np.arange(K)
    return ctr, lut


def per_frame_centres(frames, K, seed=0):
    cs = [centres_of(f, K, seed + i) for i, f in enumerate(frames)]
    return np.stack([c for c, _ in cs]), np.stack([l for _, l in cs])


def single_frame_packed(e, frames, ctrs, luts, ec, msb=True):
    """The shared-centre device call on each frame alone: (mask bits, edge bits | None, counts) of all frames, concatenated."""
    mbs, ebs, cnts = [], [], []
    for f in range(len(frames)):
        mb, eb, c = e.color_edge_packed(dev(frames[f]), ctrs[f], None if luts is None else luts[f], ec, msb_first=msb, want_counts=True)
        mbs.append(host(mb)); cnts.append(c)
        if eb is not None:
            ebs.append(host(eb))
    return np.concatenate(mbs), (np.concatenate(ebs) if ebs else None), np.concatenate(cnts)


def ec_of(ksize=3, morph_k=3, oi=1, ci=1, low=50, high=150):
    return _omni().EdgeConfig(low=low, high=high, ksize=ksize, morph_k=morph_k, open_iters=oi, close_iters=ci)


# ---- batched k-means -----------------------------------------------------------------------------------------------------------
def _kmeans_each(e, d, K, idx, attempts, seed=0):
    out = [e.kmeans_lab(d[f], K, idx, attempts=attempts, seed=seed) for f in range(d.shape[0])]
    return np.stack([c for c, _ in out]), np.array([p for _, p in out])


@pytest.mark.parametrize("sample", ["idx", "all"])
@pytest.mark.parametrize("attempts", [1, 3])
@pytest.mark.parametrize("K", [2, 8, 16, 32])
@pytest.mark.parametrize("n", [1, 3, 17])
def test_kmeans_batch_equals_single_frame_calls(eng, n, K, attempts, sample):
    h, w = 96, 120
    frames = frames_of(n, h, w, 100 * n + K, kinds=("synth", "flat", "noise"))
    idx = np.random.default_rng(42).choice(h * w, size=5000, replace=False) if sample == "idx" else None
    d = dev(frames)
    ctr, comp = eng.kmeans_lab_batch(d, K, idx, attempts=attempts, seed=5)
    want_c, want_p = _kmeans_each(eng, d, K, idx, attempts, seed=5)
    assert ctr.shape == (n, K, 3) and comp.shape == (n,)
    assert np.array_equal(ctr.view(np.uint32), want_c.view(np.uint32))       # bit for bit, NaN patterns included
    assert np.array_equal(comp, want_p)
    ctr2, comp2 = eng.kmeans_lab_batch(d, K, idx, attempts=attempts, seed=5)
    assert np.array_equal(ctr2.view(np.uint32), ctr.view(np.uint32)) and np.array_equal(comp2, comp)


def test_kmeans_batch_several_chunks_full_hd(fresh):
    """9 full-HD frames clustered on every pixel with 3 attempts need ~300 MB of runs: more than one chunk."""
    frames = frames_of(9, 1080, 1920, 7, kinds=("synth", "noise", "synth", "flat"))
    d = dev(frames)
    ctr, comp = fresh.kmeans_lab_batch(d, 8, None, attempts=3)
    want_c, want_p = _kmeans_each(fresh, d, 8, None, 3)
    assert np.array_equal(ctr.view(np.uint32), want_c.view(np.uint32)) and np.array_equal(comp, want_p)
    pick = np.random.default_rng(42).choice(1080 * 1920, size=200_000, replace=False)          # the reference's subsample
    ctr, comp = fresh.kmeans_lab_batch(d, 8, pick, attempts=3)
    want_c, want_p = _kmeans_each(fresh, d, 8, pick, 3)
    assert np.array_equal(ctr.view(np.uint32), want_c.view(np.uint32)) and np.array_equal(comp, want_p)


def test_frame_centers_gpu_mode(eng):
    from types import SimpleNamespace
    from omni_b200 import stages
    frames = frames_of(5, 500, 420, 3)                                        # 210k pixels: the seeded 200k subsample
    cfg = SimpleNamespace(color_names=["a", "b", "c", "d", "e", "f"])
    ctr, luts = stages.frame_centers(frames, cfg, mode="gpu", group=2)
    pick = np.random.default_rng(42).choice(500 * 420, size=200_000, replace=False)
    want, _ = _kmeans_each(eng, dev(frames), 6, pick, 3)
    assert np.array_equal(ctr, want)
    assert all(np.array_equal(l, stages.darkness_lut(c)[1]) for c, l in zip(ctr, luts))


# ---- per-frame packed calls ----------------------------------------------------------------------------------------------------
DEVICE_CASES = [(1, 4), (1, 16), (2, 4), (2, 8), (2, 16), (5, 4), (3, 8)]


@pytest.mark.parametrize("mode", FAMILIES)
@pytest.mark.parametrize("hw", [(67, 93), (1080, 1920)], ids=["67x93", "1080p"])
def test_device_per_frame_equals_single_frame(eng, mode, hw):
    h, w = hw
    try:
        eng.set_fast_path(mode)
        for n, K in DEVICE_CASES:
            frames = frames_of(n, h, w, n * 10 + K)
            ctrs, luts = per_frame_centres(frames, K, seed=K)
            ec = ec_of()
            for msb in (True, False):
                mb, eb, cnt = eng.color_edge_packed(dev(frames), ctrs, luts, ec, msb_first=msb, want_counts=True)
                wm, we, wc = single_frame_packed(eng, frames, ctrs, luts, ec, msb)
                assert np.array_equal(host(mb), wm), (n, K, msb)
                assert np.array_equal(host(eb), we), (n, K, msb)
                assert np.array_equal(cnt, wc), (n, K, msb)
    finally:
        eng.set_fast_path(1)


@pytest.mark.parametrize("n,K", [(1, 4), (2, 8), (5, 4), (9, 4), (9, 8), (9, 16), (5, 16)])
@pytest.mark.parametrize("hw", [(67, 93), (1080, 1920)], ids=["67x93", "1080p"])
def test_host_per_frame_equals_single_frame(eng, hw, n, K):
    """Any n: groups of 32 / K frames, the last one partial; n = 1 takes the banded single-image path at full HD."""
    h, w = hw
    frames = frames_of(n, h, w, 3 * n + K)
    ctrs, luts = per_frame_centres(frames, K, seed=n)
    ec = ec_of()
    wm, we, wc = single_frame_packed(eng, frames, ctrs, luts, ec)
    r = eng.host_color_edge_packed(frames, ctrs, luts, ec)
    assert np.array_equal(r["mask_bits"], wm) and np.array_equal(r["edge_bits"], we) and np.array_equal(r["counts"], wc)
    r = eng.host_color_edge_packed(frames, ctrs, luts, ec, msb_first=False, want_counts=False)
    wm, we, _ = single_frame_packed(eng, frames, ctrs, luts, ec, msb=False)
    assert np.array_equal(r["mask_bits"], wm) and np.array_equal(r["edge_bits"], we) and r["counts"] is None


@pytest.mark.parametrize("mode", FAMILIES)
def test_host_per_frame_every_family(eng, mode):
    frames = frames_of(9, 67, 93, 77)
    ctrs, luts = per_frame_centres(frames, 8, seed=3)
    try:
        eng.set_fast_path(mode)
        wm, we, wc = single_frame_packed(eng, frames, ctrs, luts, ec_of())
        r = eng.host_color_edge_packed(frames, ctrs, luts, ec_of())
        assert np.array_equal(r["mask_bits"], wm) and np.array_equal(r["edge_bits"], we) and np.array_equal(r["counts"], wc)
    finally:
        eng.set_fast_path(1)


STAGE03 = [dict(oi=0, ci=0), dict(oi=1, ci=1), dict(oi=2, ci=2), dict(oi=2, ci=0, morph_k=5), dict(ksize=5), None]


@pytest.mark.parametrize("prm", range(len(STAGE03)), ids=["iter0", "iter1", "iter2", "morph5", "ksize5", "colours_only"])
@pytest.mark.parametrize("hw", [(67, 93), (1080, 1920)], ids=["67x93", "1080p"])
def test_stage03_variants(eng, hw, prm):
    h, w = hw
    ec = None if STAGE03[prm] is None else ec_of(**STAGE03[prm])
    frames = frames_of(3, h, w, 40 + prm)
    ctrs, luts = per_frame_centres(frames, 8, seed=prm)
    mb, eb, cnt = eng.color_edge_packed(dev(frames), ctrs, luts, ec, want_counts=True)
    wm, we, wc = single_frame_packed(eng, frames, ctrs, luts, ec)
    assert np.array_equal(host(mb), wm) and np.array_equal(cnt, wc)
    assert (eb is None and we is None) if ec is None else np.array_equal(host(eb), we)
    frames = frames_of(5, h, w, 50 + prm)
    ctrs, luts = per_frame_centres(frames, 8, seed=prm + 1)
    r = eng.host_color_edge_packed(frames, ctrs, luts, ec)
    wm, we, wc = single_frame_packed(eng, frames, ctrs, luts, ec)
    assert np.array_equal(r["mask_bits"], wm) and np.array_equal(r["counts"], wc)
    assert (r["edge_bits"] is None) if ec is None else np.array_equal(r["edge_bits"], we)


@pytest.mark.parametrize("K", [20, 32])
def test_more_than_16_colours(eng, K):
    """K in 17..32 takes the byte-plane family frame by frame, each frame with its own centres."""
    frames = frames_of(1, 67, 93, K)
    ctrs, luts = per_frame_centres(frames, K)
    mb, eb, cnt = eng.color_edge_packed(dev(frames), ctrs, luts, ec_of(), want_counts=True)
    wm, we, wc = single_frame_packed(eng, frames, ctrs, luts, ec_of())
    assert np.array_equal(host(mb), wm) and np.array_equal(host(eb), we) and np.array_equal(cnt, wc)
    frames = frames_of(3, 67, 93, K + 1)
    ctrs, luts = per_frame_centres(frames, K)
    r = eng.host_color_edge_packed(frames, ctrs, luts, ec_of())
    wm, we, wc = single_frame_packed(eng, frames, ctrs, luts, ec_of())
    assert np.array_equal(r["mask_bits"], wm) and np.array_equal(r["edge_bits"], we) and np.array_equal(r["counts"], wc)


def test_no_lut_and_labels_above_k(eng):
    """lut None (identity per frame) and a LUT with a label >= K (no RGB-cell tables for that frame)."""
    frames = frames_of(4, 67, 93, 9)
    ctrs, luts = per_frame_centres(frames, 8)
    mb, eb = eng.color_edge_packed(dev(frames), ctrs, None, ec_of())
    wm, we, _ = single_frame_packed(eng, frames, ctrs, None, ec_of())
    assert np.array_equal(host(mb), wm) and np.array_equal(host(eb), we)
    luts[2, 3] = 20
    mb, eb = eng.color_edge_packed(dev(frames), ctrs, luts, ec_of())
    wm, we, _ = single_frame_packed(eng, frames, ctrs, luts, ec_of())
    assert np.array_equal(host(mb), wm) and np.array_equal(host(eb), we)


def test_same_centres_everywhere_is_the_shared_call(eng):
    frames = frames_of(11, 135, 250, 60)
    ctr, lut = centres_of(frames[0], 8, 1)
    ec = ec_of(low=60, high=120)
    shared = eng.host_color_edge_packed(frames, ctr, lut, ec)
    per = eng.host_color_edge_packed(frames, np.repeat(ctr[None], 11, 0), np.repeat(lut[None], 11, 0), ec)
    for k in ("mask_bits", "edge_bits", "counts"):
        assert np.array_equal(per[k], shared[k]), k
    mb, eb, cnt = eng.color_edge_packed(dev(frames[:4]), np.repeat(ctr[None], 4, 0), np.repeat(lut[None], 4, 0), ec, want_counts=True)
    assert np.array_equal(host(mb), shared["mask_bits"][:32]) and np.array_equal(host(eb), shared["edge_bits"][:32])
    assert np.array_equal(cnt, shared["counts"][:32])


def test_shard_driver_with_per_frame_centres(eng):
    from omni_b200 import batch
    frames = frames_of(6, 67, 93, 31)
    ctrs, luts = per_frame_centres(frames, 4)
    ids = batch.shard_range(6, 2, 1)
    local, r = batch.process_shard_packed(eng, frames[ids.start:ids.stop], ids, ctrs[ids.start:ids.stop], luts[ids.start:ids.stop], ec_of())
    wm, we, wc = single_frame_packed(eng, frames[ids.start:ids.stop], ctrs[ids.start:ids.stop], luts[ids.start:ids.stop], ec_of())
    assert sorted(local) == list(ids) and np.array_equal(r["mask_bits"], wm) and np.array_equal(r["edge_bits"], we)
    assert all(np.array_equal(local[f], wc[j * 4:(j + 1) * 4]) for j, f in enumerate(ids))


# ---- call order and the candidate-table cache ------------------------------------------------------------------------------------
def _per_frame_call(e, frames, ctrs, luts, ec):
    mb, eb, c = e.color_edge_packed(dev(frames), ctrs, luts, ec, want_counts=True)
    return host(mb), host(eb), c


def _shared_call(e, frames, ctr, lut, ec):
    r = e.host_color_edge_packed(frames, ctr, lut, ec)
    return r["mask_bits"], r["edge_bits"], r["counts"]


@pytest.mark.parametrize("cache", [True, False])
@pytest.mark.parametrize("hw", [(67, 93), (720, 1280)], ids=["67x93", "720p"])
def test_call_order_and_table_cache(hw, cache):
    """A per-frame call followed by shared-centre calls on one context, and the reverse, give the bytes of fresh contexts.  The
    shared centres are those of the per-frame call's last frame (a table-cache hit is correct), of its first frame (the cache
    must rebuild), and new ones."""
    omni = _omni()
    h, w = hw
    frames = frames_of(4, h, w, 90)
    ctrs, luts = per_frame_centres(frames, 8, seed=4)
    ec = ec_of()
    sets = [(ctrs[3], luts[3]), (ctrs[0], luts[0]), centres_of(frames[1], 8, 99)]

    def on_fresh(fn, *a):
        e = omni.Engine(0)
        try:
            e.set_table_cache(cache)
            return fn(e, *a)
        finally:
            e.close()

    want_pf = on_fresh(_per_frame_call, frames, ctrs, luts, ec)
    want_sh = [on_fresh(_shared_call, frames, c, l, ec) for c, l in sets]
    for order in ("per_frame_first", "shared_first"):
        e = omni.Engine(0)
        try:
            e.set_table_cache(cache)
            got_sh = []
            if order == "shared_first":
                got_sh = [_shared_call(e, frames, c, l, ec) for c, l in sets]
            got_pf = _per_frame_call(e, frames, ctrs, luts, ec)
            if order == "per_frame_first":
                got_sh = [_shared_call(e, frames, c, l, ec) for c, l in sets]
            got_pf2 = _per_frame_call(e, frames, ctrs, luts, ec)
        finally:
            e.close()
        for a, b in zip(got_pf + got_pf2, want_pf + want_pf):
            assert np.array_equal(a, b), order
        for got, want in zip(got_sh, want_sh):
            for a, b in zip(got, want):
                assert np.array_equal(a, b), order


# ---- argument errors ----------------------------------------------------------------------------------------------------------
def test_argument_errors(eng):
    omni = _omni()
    L, capi = omni.capi.lib(), omni.capi
    frames = frames_of(3, 67, 93, 5)
    d = dev(frames)
    n, h, w = 3, 67, 93
    rb = (w + 7) // 8
    K = 8
    ctrs, luts = per_frame_centres(frames, K)
    mb = torch.empty((n * K, h, rb), dtype=torch.uint8, device="cuda")
    eb = torch.empty_like(mb)
    p = ec_of().to_c()
    f32p, u8p = C.POINTER(C.c_float), C.POINTER(C.c_uint8)

    def dev_call(ctr, lut, nf=n, k=K):
        return L.omni_color_edge_packed_frames(eng._h, d.data_ptr(), nf, d.stride(0), h, w, d.stride(1),
                                               ctr.ctypes.data_as(f32p) if ctr is not None else None, k,
                                               lut.ctypes.data_as(u8p) if lut is not None else None, C.byref(p),
                                               mb.data_ptr(), mb.stride(0), mb.stride(1), eb.data_ptr(), eb.stride(0), eb.stride(1),
                                               capi.BITS_MSB_FIRST, None, None)

    def host_call(ctr, lut):
        hm = np.empty((n * K, h, rb), np.uint8)
        he = np.empty_like(hm)
        return L.omni_host_color_edge_packed_frames(eng._h, frames.ctypes.data, n, frames.strides[0], h, w, frames.strides[1],
                                                    ctr.ctypes.data_as(f32p) if ctr is not None else None, K,
                                                    lut.ctypes.data_as(u8p) if lut is not None else None, C.byref(p),
                                                    hm.ctypes.data, hm.strides[0], hm.strides[1], he.ctypes.data, he.strides[0],
                                                    he.strides[1], capi.BITS_MSB_FIRST, None)

    def err():
        return L.omni_last_error_string().decode()

    assert dev_call(ctrs, luts) == 0 and host_call(ctrs, luts) == 0
    assert dev_call(None, luts) == -1 and "NULL" in err()
    assert host_call(None, luts) == -1 and err()
    bad = luts.copy()
    bad[2, 5] = 40                                                            # frame 2's LUT: label 40 >= OMNI_MAX_K
    assert dev_call(ctrs, bad) == -1 and "lut" in err()
    assert host_call(ctrs, bad) == -1 and "lut" in err()
    assert dev_call(np.ascontiguousarray(np.concatenate([ctrs, ctrs[:2]])), np.concatenate([luts, luts[:2]]), nf=5) == -1
    assert "exceeds" in err()                                                 # 5 * 8 planes > 32 in the device form
    with pytest.raises(ValueError):
        eng.color_edge_packed(d, ctrs[:2], luts[:2], ec_of())                 # centres of 2 frames for 3 frames
    with pytest.raises(ValueError):
        eng.host_color_edge_packed(frames, ctrs, luts[:, :4], ec_of())
    with pytest.raises(omni.OmniError):
        eng.kmeans_lab_batch(d, 0, None)
    idx = np.array([0, h * w], np.int32)
    with pytest.raises(omni.OmniError, match="out of range"):
        eng.kmeans_lab_batch(d, 2, idx)
