"""The rule the GPU tracer numbers components by (csrc/trace.cu): cv2.connectedComponentsWithStats(S, connectivity=8) labels
components in the order of the first 2x2 BLOCK, in block-raster order, that holds one of their pixels -- block key
(y >> 1) * ceil(w / 2) + (x >> 1) -- not in pixel-raster order.  Pinned here against cv2 itself, including odd widths and
images of 2048^2 and more (cv2's threaded path)."""
import cv2
import numpy as np
import pytest
from scipy import ndimage


def _block_rank_labels(S):
    """NumPy restatement: 8-connected components (scipy), numbered by the rank of their minimum block key."""
    lab, n = ndimage.label(S, structure=np.ones((3, 3), int))
    if n == 0:
        return lab
    ys, xs = np.nonzero(lab)
    key = (ys // 2).astype(np.int64) * ((S.shape[1] + 1) // 2) + xs // 2
    first = np.full(n + 1, np.iinfo(np.int64).max)
    np.minimum.at(first, lab[ys, xs], key)
    rank = np.empty(n + 1, np.int64)
    rank[0] = 0
    rank[1 + np.argsort(first[1:], kind="stable")] = np.arange(1, n + 1)
    return rank[lab]


CASES = [((37, 41), 0.05), ((1, 97), 0.3), ((97, 1), 0.3), ((2, 2), 0.5), ((63, 255), 0.2), ((512, 701), 0.1),
         ((1024, 1023), 0.4), ((2048, 2048), 0.05), ((2048, 2049), 0.2), ((2304, 2048), 0.35)]


@pytest.mark.parametrize("shape,p", CASES)
def test_cv2_labels_follow_block_order(shape, p):
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    S = (rng.random(shape) < p).astype(np.uint8)
    num, lab, _st, _c = cv2.connectedComponentsWithStats(S, connectivity=8)
    want = _block_rank_labels(S)
    assert num - 1 == int(want.max())
    assert np.array_equal(lab, want)


def test_pixel_raster_order_is_not_the_rule():
    """Components whose pixels come first in raster order but whose blocks come later get the later label."""
    S = np.zeros((4, 8), np.uint8)
    S[1, 0] = 1          # (x 0, y 1): block key 0
    S[0, 5] = 1          # (x 5, y 0): first in raster order, block key 2
    S[3, 1] = 1          # (x 1, y 3): block key 4
    num, lab, _st, _c = cv2.connectedComponentsWithStats(S, connectivity=8)
    assert num == 4 and lab[1, 0] == 1 and lab[0, 5] == 2 and lab[3, 1] == 3
    assert np.array_equal(lab, _block_rank_labels(S))
