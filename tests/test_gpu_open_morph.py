"""The fused label-domain open + morphology kernel (fk_open_morph) at the geometry its shared-memory staging has to get right:
the clipped column groups of 30 words at the left / right image border, strips cut by the image bottom, images smaller than one
strip, plane groups of one frame (K up to 16, frame batches of n * K = 32), strided outputs, the colours-only call and the four
stage-03 morphology kinds.  Masks, edges and packed bits are compared bit for bit with the round-1 family
(omni_set_fast_path 3) and with the oracle.  Needs a B200: `-m gpu`."""
import numpy as np
import pytest

from helpers import synth, uniform_img

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def eng():
    import omni_b200
    e = omni_b200.Engine(0)
    yield e
    e.set_fast_path(1)
    e.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def host(t):
    return t.cpu().numpy()


def _image(h, w, K, seed=0):
    from oracle import refport as rp
    img = synth(h, w, seed + K + w, cell=16) if min(h, w) >= 16 else uniform_img(h, w, seed + K)
    if h * w >= 4 * K:
        ctr = rp.kmeans_lab_centers(img, K)
    else:
        ctr = np.random.default_rng(seed + 1).random((K, 3)).astype(np.float32) * 255
    _o, lut = rp.darkness_order(ctr)
    return img, ctr, lut.astype(np.uint8)


def _oracle(img, ctr, lut, K, mk, oi, ci):
    from oracle import cmodel as cm
    raw = cm.assign_f32(cm.bgr2lab(img), ctr)
    wm = cm.layer_masks(raw, K, lut)
    we = np.stack([cm.edge_chain(m, mk, oi, ci, 3, 50, 150) for m in wm])
    return wm, we


def _both_families(eng, fn):
    """fn() under the label pipeline (mode 1) and the round-1 family (mode 3)."""
    try:
        eng.set_fast_path(1)
        new = fn()
        eng.set_fast_path(3)
        old = fn()
    finally:
        eng.set_fast_path(1)
    return new, old


def _check(eng, h, w, K, mk=3, oi=1, ci=1, oracle=True):
    import omni_b200
    img, ctr, lut = _image(h, w, K)
    ec = omni_b200.EdgeConfig(morph_k=mk, open_iters=oi, close_iters=ci)
    d = dev(img)

    def run():
        _l, m, e = eng.color_edge(d, ctr, lut, ec)
        mb, eb = eng.color_edge_packed(d, ctr, lut, ec)
        cb, _none = eng.color_edge_packed(d, ctr, lut, None)
        return host(m), host(e), host(mb), host(eb), host(cb)

    (m, e, mb, eb, cb), old = _both_families(eng, run)
    for a, b in zip((m, e, mb, eb, cb), old):
        assert np.array_equal(a, b)
    assert np.array_equal(mb, np.packbits(m > 0, axis=2)) and np.array_equal(cb, mb)
    assert np.array_equal(eb, np.packbits(e > 0, axis=2))
    if oracle:
        wm, we = _oracle(img, ctr, lut, K, mk, oi, ci)
        assert np.array_equal(m, wm)
        assert np.array_equal(e, we)


# w % 32 in {0, 1, 2, 31}; just over 1, 2 column groups (960 px = 30 words); heights below / just above one strip
@pytest.mark.parametrize("h,w", [(40, 64), (40, 65), (40, 66), (40, 95), (20, 961), (33, 962), (57, 1921), (65, 1000),
                                 (130, 990), (31, 1919)])
@pytest.mark.parametrize("K", [3, 16])
def test_column_groups_and_strips(eng, h, w, K):
    _check(eng, h, w, K)


@pytest.mark.parametrize("h,w", [(1, 1), (1, 2), (2, 1), (2, 3), (3, 3), (1, 40), (3, 40), (40, 3), (2, 33)])
def test_tiny_images(eng, h, w):
    _check(eng, h, w, 2)


@pytest.mark.parametrize("K", [2, 3, 8, 15, 16])
def test_plane_groups(eng, K):
    _check(eng, 150, 1000, K)


@pytest.mark.parametrize("mk,oi,ci", [(3, 0, 0), (3, 1, 0), (3, 0, 1), (3, 1, 1), (1, 1, 1)],
                         ids=["kind0", "kind1", "kind2", "kind3", "morph_k1"])
def test_morphology_kinds(eng, mk, oi, ci):
    _check(eng, 97, 1925, 8, mk, oi, ci)


@pytest.mark.parametrize("n,K,hw", [(2, 16, (70, 1000)), (4, 8, (65, 97)), (16, 2, (9, 40))])
def test_frame_batches_of_32_planes(eng, n, K, hw):
    """n * K = 32 planes in one launch: every frame as its own call, and the round-1 family's batch."""
    import omni_b200
    frames = np.stack([synth(hw[0], hw[1], 70 + f, cell=16) for f in range(n)])
    _img, ctr, lut = _image(hw[0], hw[1], K)
    ec = omni_b200.EdgeConfig()
    d = dev(frames)

    def run():
        m = torch.full((n, K) + hw, 9, dtype=torch.uint8, device="cuda")
        e = torch.full((n, K) + hw, 9, dtype=torch.uint8, device="cuda")
        eng.color_edge_batch(d, ctr, lut, ec, masks=m, edges=e)
        return host(m), host(e)

    (m, e), (m3, e3) = _both_families(eng, run)
    assert np.array_equal(m, m3) and np.array_equal(e, e3)
    for f in range(n):
        _l, mf, ef = eng.color_edge(d[f], ctr, lut, ec)
        assert np.array_equal(m[f], host(mf)) and np.array_equal(e[f], host(ef)), f
    wm, we = _oracle(frames[-1], ctr, lut, K, 3, 1, 1)
    assert np.array_equal(m[-1], wm) and np.array_equal(e[-1], we)


def test_strided_outputs(eng):
    """Masks and edges written into views with row and plane gaps: the bytes around the views stay untouched."""
    import omni_b200
    h, w, K = 75, 1001, 8
    img, ctr, lut = _image(h, w, K)
    ec = omni_b200.EdgeConfig()
    d = dev(img)
    _l, m_ref, e_ref = eng.color_edge(d, ctr, lut, ec)
    bm = torch.full((K + 1, h + 7, w + 45), 7, dtype=torch.uint8, device="cuda")
    be = torch.full((K + 1, h + 7, w + 45), 7, dtype=torch.uint8, device="cuda")
    vm, ve = bm[1:, 3:3 + h, 13:13 + w], be[1:, 3:3 + h, 13:13 + w]
    eng.color_edge(d, ctr, lut, ec, masks=vm, edges=ve)
    assert torch.equal(vm, m_ref) and torch.equal(ve, e_ref)
    for b in (bm, be):
        outside = b.clone()
        outside[1:, 3:3 + h, 13:13 + w] = 7
        assert bool((outside == 7).all())
