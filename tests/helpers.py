"""Shared test helpers: synthetic inputs (SURVEY.md 8d generator) and golden-case loading."""
import json
import os

import cv2
import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PIPE_CASES = ["pipe_default_k4", "pipe_treecfg_k4", "pipe_k8_2to1"]


def synth(H, W, seed, cell=32):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (max(1, H // cell), max(1, W // cell), 3), np.uint8)
    img = cv2.resize(base, (W, H), interpolation=cv2.INTER_CUBIC)
    noise = rng.integers(-12, 13, img.shape, dtype=np.int16)
    return np.clip(img.astype(np.int16) + noise, 0, 255).astype(np.uint8)


def uniform_img(H, W, seed):
    return np.random.default_rng(seed).integers(0, 256, (H, W, 3), dtype=np.uint8)


KMEANS_TOL = 0.02          # k-means quality bound: compactness within 2 % of cv2.kmeans' on the same sample


def lab_sample(img, limit=200_000):
    """02_color_extract.py:35-42: the seeded subsample (None: every pixel) and its 8-bit Lab values from cv2."""
    n = img.shape[0] * img.shape[1]
    idx = np.random.default_rng(42).choice(n, size=limit, replace=False) if n > limit else None
    flat = img.reshape(-1, 3) if idx is None else img.reshape(-1, 3)[idx]
    lab = cv2.cvtColor(np.ascontiguousarray(flat).reshape(-1, 1, 3), cv2.COLOR_BGR2LAB).reshape(-1, 3).astype(np.float32)
    return idx, lab


def compactness(lab, centers):
    """Sum over the samples of the squared distance to the nearest centre, in float64."""
    d = ((lab[:, None, :].astype(np.float64) - centers[None].astype(np.float64)) ** 2).sum(axis=2)
    return float(d.min(axis=1).sum())


def smooth_u8(H, W, seed, k=7):
    g = np.random.default_rng(seed).integers(0, 256, (H + 2 * k, W + 2 * k), dtype=np.uint8)
    return np.ascontiguousarray(cv2.GaussianBlur(g, (k, k), 0)[k:k + H, k:k + W])


def blob_mask(H, W, seed, p=0.5, k=9):
    """Binary {0,255} mask with blobby regions (threshold of smoothed noise)."""
    s = smooth_u8(H, W, seed, k)
    return ((s > np.quantile(s, 1 - p)) * 255).astype(np.uint8)


# dataclass defaults of the keys stages 01-03 read (reference config.py:14-36); a pre-seeded
# config.json only holds the keys it was seeded with, load_config fills the rest from these
CFG_DEFAULTS = {
    "max_dimension": 2000,
    "color_names": ["layer_dark", "layer_mid", "layer_skin", "layer_light"],
    "colors": [[0, 0, 0], [255, 0, 0], [0, 255, 0], [0, 0, 255]],
    "edge_low_threshold": 50, "edge_high_threshold": 150, "edge_kernel_size": 3,
    "edge_morph_kernel": 3, "edge_morph_open_iters": 1, "edge_morph_close_iters": 1,
}


def load_pipe_case(name):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    meta = json.load(open(os.path.join(GOLDEN, name + ".json")))
    meta["config"] = {**CFG_DEFAULTS, **meta["config"]}
    return z, meta


def plane_of_name(names):
    """02_color_extract.py:130-133: names sorted by darkness rank (stable) get planes 0..K-1."""
    def rank(n):
        s = n.lower()
        for key, r in (("dark", 0), ("mid", 1), ("skin", 2), ("light", 3)):
            if key in s:
                return r
        return 2
    order = sorted(names, key=rank)
    return {n: order.index(n) for n in names}
