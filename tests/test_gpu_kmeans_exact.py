"""The device k-means (omni_kmeans_lab / omni_kmeans_lab_batch, csrc/kmeans.cu) against oracle/kmeans_model.py, bit for bit: the
float32 centres and the compactness must equal the model's exactly.  The kernel is built with --fmad=false, sums integers and
keeps the compactness in fixed point, so there is no tolerance to hide a wrong tie rule, an off-by-one in the seeding's thread
ranges, stale run state across chunks of a batch or an empty cluster that loses its centre.  Needs a B200: `-m gpu`."""
import numpy as np
import pytest

from helpers import synth, uniform_img
from oracle import kmeans_model as km

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def eng():
    import omni_b200
    e = omni_b200.Engine(0)
    yield e
    e.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_same(got, want):
    (gc, gp), (wc, wp) = got, want
    assert gc.shape == wc.shape
    assert np.array_equal(gc.view(np.uint32), wc.view(np.uint32)), (gc, wc)
    assert np.array_equal(gp, wp), (gp, wp)


def check(eng, img, K, idx=None, **kw):
    assert_same(eng.kmeans_lab(dev(img), K, idx, **kw), km.kmeans_lab(img, K, idx, **kw))


def pick200k(img):
    from omni_b200.stages import _sample_pick
    return _sample_pick(img.shape[0] * img.shape[1], 200_000)


def palette_img(bgr, h, w, seed):
    """h x w pixels of the given BGR colours in a seeded random arrangement, each colour (nearly) equally often."""
    bgr = np.asarray(bgr, np.uint8)
    which = np.random.default_rng(seed).permutation(np.arange(h * w) % len(bgr))
    return bgr[which].reshape(h, w, 3)


GREYS = [(v, v, v) for v in range(100, 106)]     # 8-bit Lab L = 108 .. 113, a = b = 128: half-integer means, tied assignments


# ---- the reference's use: its seeded 200k subsample, 3 attempts, 40 iterations, eps 0.5 ------------------------------------------
@pytest.mark.parametrize("K", [2, 3, 4, 8, 16, 32])
def test_reference_subsample(eng, K):
    img = synth(500, 640, K)
    check(eng, img, K, pick200k(img))


# ---- criteria ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw", [(300, 400), (480, 520)], ids=["120k", "250k"])
def test_every_pixel(eng, hw):
    check(eng, synth(hw[0], hw[1], 11), 8)


@pytest.mark.parametrize("kw", [dict(max_iter=1), dict(max_iter=2), dict(eps=0.0, max_iter=60), dict(eps=1.0e6),
                                dict(attempts=1), dict(attempts=2)],
                         ids=["iter1", "iter2", "eps0", "eps_large", "attempts1", "attempts2"])
def test_criteria(eng, kw):
    img = synth(240, 320, 21)
    check(eng, img, 6, np.random.default_rng(5).choice(240 * 320, 30_000, replace=False), **kw)


def test_64_attempts(eng):
    check(eng, synth(100, 120, 22), 5, attempts=64)


@pytest.mark.parametrize("seed", [1, 12345, 2 ** 32 + 7, 2 ** 63 + 11, 2 ** 64 - 1])
def test_seeds(eng, seed):
    check(eng, synth(160, 200, 23), 4, seed=seed)


# ---- ties and degenerate data -----------------------------------------------------------------------------------------------------
def test_flat_image(eng):
    """total == 0 from the second centre on (the draw's fallbacks decide), and every attempt ties."""
    check(eng, np.full((48, 70, 3), (40, 170, 220), np.uint8), 4)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
@pytest.mark.parametrize("ncol", [2, 3])
def test_fewer_colours_than_centres(eng, ncol, seed):
    """Duplicate centres, empty clusters, and attempts of equal compactness whose centres come in different orders.  Once every
    colour is a centre the draw has total == 0 and falls back to thread 1023's range: with n = 2048 that is samples 2046 and
    2047, given different colours here, so the fallback's choice of the last one shows in the duplicate centres."""
    cols = np.array([(20, 20, 200), (240, 200, 10), (90, 140, 60)][:ncol], np.uint8)
    img = np.random.default_rng(seed).choice(cols, size=(32, 64))
    img[31, 62], img[31, 63] = cols[seed % ncol], cols[(seed + 1) % ncol]
    check(eng, img, 8, seed=seed)
    check(eng, img, 8, seed=seed, attempts=8)


def test_as_many_samples_as_centres(eng):
    img = uniform_img(30, 40, 3)
    idx = np.random.default_rng(3).choice(1200, 16, replace=False)
    check(eng, img, 16, idx)
    check(eng, img, 4, np.full(4, 77))                                # n == K, all one sample
    check(eng, img, 6, np.random.default_rng(4).integers(0, 1200, 5000))   # indices that repeat


@pytest.mark.parametrize("seed", range(8))
def test_grey_ramp_ties(eng, seed):
    """Six grey levels of consecutive L: centres at half-integers and samples exactly between two of them, and seeding
    candidates of different colours with equal potential."""
    img = palette_img(GREYS, 36, 50, seed)
    check(eng, img, 2, seed=seed, attempts=1)
    check(eng, img, 3, seed=seed)
    check(eng, palette_img(GREYS[::2], 36, 50, seed), 2, seed=seed, attempts=1)


# ---- geometry ---------------------------------------------------------------------------------------------------------------------
def test_strips(eng):
    for w in range(1, 9):
        img = uniform_img(1, w, w)
        for K in sorted({1, (w + 1) // 2, w}):
            check(eng, img, K)


@pytest.mark.parametrize("n", [1023, 1024, 1025, 2047, 2048, 2049, 3 * 1024])
def test_seeding_thread_ranges(eng, n):
    """Sample counts around the seeding's split into 1024 thread ranges of ceil(n / 1024) samples."""
    img = synth(60, 80, n)
    check(eng, img, 6, np.random.default_rng(n).choice(60 * 80, n, replace=False), max_iter=4)


def test_crop_with_wide_pitch(eng):
    big = synth(300, 500, 31)
    crop = big[37:237, 91:341]                                       # pitch 1500 > 3 * 250
    d = dev(big)[37:237, 91:341]
    assert d.stride(0) == 1500
    for idx in (None, np.random.default_rng(6).choice(200 * 250, 20_000, replace=False)):
        assert_same(eng.kmeans_lab(d, 5, idx), km.kmeans_lab(crop, 5, idx))


def _near_white(h, w, seed):
    """White (8-bit Lab L = 255) but for one pixel in 64 a little darker: the integer sums come within 0.4 % of 2^32."""
    img = np.full((h, w, 3), 255, np.uint8)
    rng = np.random.default_rng(seed)
    dark = rng.random((h, w)) < 1 / 64
    img[dark] = rng.integers(235, 255, (int(dark.sum()), 3), dtype=np.uint8)
    return img


def test_largest_sample(eng):
    """4096 x 4096 in every-pixel mode: n = 2^24, the most the u32 accumulators allow."""
    img = _near_white(4096, 4096, 41)
    d = dev(img)
    for K in (1, 2):
        assert_same(eng.kmeans_lab(d, K, None, attempts=1, max_iter=2), km.kmeans_lab(img, K, None, attempts=1, max_iter=2))
    import omni_b200
    with pytest.raises(omni_b200.OmniError):
        eng.kmeans_lab(torch.zeros((4097, 4096, 3), dtype=torch.uint8, device="cuda"), 2)


# ---- batches: the chunking must not show ------------------------------------------------------------------------------------------
def test_batch_of_tiny_frames_64_attempts(eng):
    """1025 frames of 8 x 8 with 64 attempts: chunks of 65535 / 64 = 1023 frames, the second one partial."""
    rng = np.random.default_rng(51)
    frames = rng.integers(0, 256, (1025, 8, 8, 3), dtype=np.uint8)
    frames[1::7] = frames[1::7, :1, :1]                              # some flat frames
    frames[2::7] = palette_img([(0, 0, 0), (255, 255, 255), (0, 0, 255)], 8, 8, 1)
    got = eng.kmeans_lab_batch(dev(frames), 4, None, attempts=64)
    assert_same(got, km.kmeans_lab_batch(frames, 4, None, attempts=64))


def test_batch_of_full_hd_frames(eng):
    """11 frames of 1080p on every pixel with 2 attempts need 25 MB each: more than one 256 MiB chunk."""
    frames = np.stack([synth(1080, 1920, 60 + i, cell=16) for i in range(11)])
    got = eng.kmeans_lab_batch(dev(frames), 4, None, attempts=2, max_iter=6)
    for f in (0, 10):
        assert_same((got[0][f], got[1][f]), km.kmeans_lab(frames[f], 4, None, attempts=2, max_iter=6))


# ---- argument errors --------------------------------------------------------------------------------------------------------------
def test_argument_errors_leave_the_context_usable(eng):
    import omni_b200
    img = synth(20, 30, 71)
    d = dev(img)
    bad = [dict(K=3, attempts=0), dict(K=3, attempts=65), dict(K=3, max_iter=0), dict(K=3, max_iter=1001), dict(K=3, eps=-0.5),
           dict(K=3, sample_idx=np.arange(2)), dict(K=3, sample_idx=np.array([0, 600])), dict(K=3, sample_idx=np.array([5, -1, 7]))]
    for kw in bad:
        with pytest.raises(omni_b200.OmniError):
            eng.kmeans_lab(d, **kw)
    with pytest.raises(omni_b200.OmniError):
        eng.kmeans_lab(dev(img[:4, :5]), 21)                          # K > n in every-pixel mode
    check(eng, img, 3)
