"""NumPy restatement of the device k-means (omnirevolve-image-processor_b200/csrc/kmeans.cu) -- TEST INFRASTRUCTURE ONLY.

It gives the kernel's centres and compactness bit for bit, which is possible because of how the kernel computes:
  - the library is built with --fmad=false, so every float32 product and sum rounds on its own, as NumPy float32 does;
  - in the seeding every distance is an integer below 2^24 and every double sum an integer below 2^53, so no order of summation
    changes a bit (the model sums integers);
  - the Lloyd sums are u32 integers, the compactness a u64 in 1/1024 units, and the RNG a pure function of (seed, attempt, k, t).
So this is the kernel's algorithm step for step, not a textbook k-means: the two-level search of the seeding draw over 1024 thread
ranges, its fallbacks, the strict-< tie rules and the fixed-point compactness are all part of the result.

The assignment of a sample depends only on its value, so the Lloyd steps run on the distinct Lab values of a frame weighted by
their counts; the integer sums are the same as over every sample.  A batch is one independent model run per frame: the kernel
groups frames into chunks, and that must not show in its results.  tests/test_gpu_kmeans_exact.py compares the two.
"""
import numpy as np

from . import cmodel

SEED_THREADS = 1024                      # KM_SEED_THREADS: the coarse level of the seeding draw
TRIALS = 3                               # KM_TRIALS: candidates per new centre
FIX = np.float32(1024.0)                 # KM_FIX: compactness in 1/1024 units
MAX_K = 32
M64 = (1 << 64) - 1


def km_mix(x: int) -> int:
    x = (x + 0x9E3779B97F4A7C15) & M64
    x = ((x ^ (x >> 30)) * 0xBF58476D1CE4E5B9) & M64
    x = ((x ^ (x >> 27)) * 0x94D049BB133111EB) & M64
    return x ^ (x >> 31)


def km_uniform(seed: int, a: int, b: int, c: int) -> float:
    """Uniform in [0, 1) from 53 bits of km_mix(seed ^ km_mix(a << 40 ^ b << 20 ^ c))."""
    r = km_mix((seed & M64) ^ km_mix(((a << 40) ^ (b << 20) ^ c) & M64))
    return float(r >> 11) * 2.0 ** -53


def lab_samples(frames: np.ndarray, idx=None) -> np.ndarray:
    """fk_km_gather: the 8-bit Lab values (int32 [F, n, 3]) of pixel idx[i] of every frame (idx None: pixel i).  frames: [F, H, W, 3]
    BGR, any strides (a crop of a wider image has pitch > 3 * w)."""
    flat = np.asarray(frames).reshape(frames.shape[0], -1, 3)
    if idx is not None:
        flat = flat[:, np.asarray(idx, dtype=np.int64)]
    return cmodel.bgr2lab(flat).astype(np.int32)


def _d2_int(s: np.ndarray, c: np.ndarray) -> np.ndarray:
    """km_d2 of the integer samples s [n, 3] to integer centres c [R, 3] -> [R, n]: exact in float32, so computed on integers."""
    out = np.zeros((c.shape[0], s.shape[0]), np.int32)
    for ch in range(3):
        d = s[None, :, ch] - c[:, ch, None]
        out += d * d
    return out


def seed_centres(s: np.ndarray, K: int, attempts: int, seed: int) -> np.ndarray:
    """fk_km_seed for every attempt of one frame: float32 [attempts, K, 3].  s: int32 [n, 3]."""
    n = s.shape[0]
    per = (n + SEED_THREADS - 1) // SEED_THREADS  # thread t sums the samples [t * per, (t + 1) * per)
    starts = np.arange(0, n, per)                  # threads with a non-empty range; the others add 0 to every sum
    A = attempts
    rows = np.arange(A)
    first = [min(n - 1, int(km_uniform(seed, a, 0, 0) * n)) for a in range(A)]
    ctr = np.zeros((A, K, 3), np.int32)
    ctr[:, 0] = s[first]
    dist = _d2_int(s, ctr[:, 0])                   # [A, n]
    win = np.arange(per)
    for k in range(1, K):
        cum = np.cumsum(np.add.reduceat(dist, starts, axis=1, dtype=np.int64), axis=1).astype(np.float64)  # exact: < 2^53
        total = cum[:, -1]
        r = np.array([[km_uniform(seed, a, k, t + 1) for t in range(TRIALS)] for a in range(A)]) * total[:, None]
        # coarse level: the first thread whose cumulative sum exceeds r, acc = the sum before it; none (total == 0, r == 0):
        # thread 1023, acc = the whole sum
        th = (cum[:, None, :] <= r[:, :, None]).sum(axis=2)
        found = th < len(starts)
        before = np.where(th > 0, np.take_along_axis(cum, np.maximum(th - 1, 0), axis=1), 0.0)
        acc = np.where(found, before, total[:, None])
        th = np.where(found, th, SEED_THREADS - 1)
        a = np.minimum(n, th * per)
        b = np.minimum(n, a + per)
        # fine level: the first sample of that thread's range at which the running sum exceeds r; none: max(a, b - 1)
        pos = a[..., None] + win
        inside = pos < b[..., None]
        vals = np.take_along_axis(dist, np.minimum(pos, n - 1).reshape(A, -1), axis=1).reshape(pos.shape)
        run = acc[..., None] + np.cumsum(np.where(inside, vals, 0), axis=2, dtype=np.int64).astype(np.float64)
        over = (run > r[..., None]) & inside
        pick = np.where(over.any(axis=2), a + np.argmax(over, axis=2), np.maximum(a, b - 1))
        pick = np.clip(pick, 0, n - 1)
        # the candidate of least potential (strict <: the lowest of equal ones)
        pot = np.stack([np.minimum(dist, _d2_int(s, s[pick[:, t]])).sum(axis=1, dtype=np.int64) for t in range(TRIALS)], axis=1)
        bt = np.argmin(pot, axis=1)
        ctr[:, k] = s[pick[rows, bt]]
        dist = np.minimum(dist, _d2_int(s, ctr[:, k]))
    return ctr.astype(np.float32)


def _assign(u: np.ndarray, w: np.ndarray, ctr: np.ndarray):
    """fk_km_assign for runs ctr [R, K, 3] over the distinct values u (int32 [m, 3]) with counts w: (sums int64 [R, K, 3],
    counts int64 [R, K], compactness int [R] in 1/1024 units)."""
    R, K, _ = ctr.shape
    uf = [np.ascontiguousarray(u[:, ch], dtype=np.float32) for ch in range(3)]
    bd = np.full((R, u.shape[0]), np.float32(3.0e38), np.float32)
    best = np.zeros((R, u.shape[0]), np.int32)
    d, t = np.empty_like(bd), np.empty_like(bd)
    closer = np.empty(bd.shape, bool)
    for k in range(K):                             # float32, each operation rounded: (d0 * d0 + d1 * d1) + d2 * d2
        np.subtract(uf[0], ctr[:, k, 0, None], out=d)
        d *= d
        for ch in (1, 2):
            np.subtract(uf[ch], ctr[:, k, ch, None], out=t)
            t *= t
            d += t
        np.less(d, bd, out=closer)                 # strict <: the first minimum
        np.minimum(d, bd, out=bd)
        np.putmask(best, closer, k)
    term = (bd * FIX + np.float32(0.5)).astype(np.uint64).astype(np.int64)
    comp = (term * w).sum(axis=1)
    best += K * np.arange(R, dtype=np.int32)[:, None]
    bins = best.ravel()
    # float64 bincount is exact here: every sum is an integer below 2^32 (n <= 2^24 samples of at most 255)
    sums = np.stack([np.bincount(bins, weights=np.tile(wv, R), minlength=R * K)
                     for wv in (w * u[:, 0], w * u[:, 1], w * u[:, 2], w)], axis=1).reshape(R, K, 4).astype(np.int64)
    return sums[..., :3], sums[..., 3], comp


def _update(ctr: np.ndarray, sums: np.ndarray, cnt: np.ndarray, eps2: np.float32):
    """fk_km_update: (new centres, converged [R]).  c = f32(f64(sum) / f64(cnt)); an empty cluster keeps its centre; the shift is
    the largest float32 squared move."""
    full = cnt > 0
    mean = (sums / np.maximum(cnt, 1)[..., None]).astype(np.float32)
    new = np.where(full[..., None], mean, ctr)
    dd = new - ctr
    sq = dd * dd
    shift = ((sq[..., 0] + sq[..., 1]) + sq[..., 2]).max(axis=1)
    return new, shift <= eps2


def kmeans_frame(s: np.ndarray, K: int, attempts: int = 3, max_iter: int = 40, eps: float = 0.5, seed: int = 0):
    """All attempts of one frame's samples s (int32 [n, 3]): (centres float32 [K, 3], compactness)."""
    ctr = seed_centres(s, K, attempts, seed)
    packed = s[:, 0] | (s[:, 1] << 8) | (s[:, 2] << 16)
    vals, w = np.unique(packed, return_counts=True)
    u = np.stack([vals & 255, (vals >> 8) & 255, vals >> 16], axis=1).astype(np.int32)
    w = w.astype(np.int64)
    eps2 = np.float32(np.float32(eps) * np.float32(eps))
    live = np.ones(attempts, bool)
    for _ in range(max_iter):
        if not live.any():
            break
        sums, cnt, _comp = _assign(u, w, ctr[live])
        ctr[live], conv = _update(ctr[live], sums, cnt, eps2)
        live[np.flatnonzero(live)[conv]] = False
    _s, _c, comp = _assign(u, w, ctr)              # the forced pass: compactness of the final centres
    ba = int(np.argmin(comp))                      # fk_km_keep_best: the first strictly smallest
    return ctr[ba].copy(), int(comp[ba]) / 1024.0


def _check(n, npix, idx, K, attempts, max_iter, eps):
    """The argument domain of omni_kmeans_lab (capi.cu kmeans_checked)."""
    if not (1 <= K <= MAX_K and 1 <= attempts <= 64 and 1 <= max_iter <= 1000 and eps >= 0 and K <= n <= (1 << 24)):
        raise ValueError(f"k-means arguments outside the kernel's domain: n={n} K={K} attempts={attempts} max_iter={max_iter} eps={eps}")
    if idx is not None and not ((np.asarray(idx) >= 0) & (np.asarray(idx) < npix)).all():
        raise ValueError("sample index out of range")


def kmeans_lab_batch(frames, K: int, sample_idx=None, attempts: int = 3, max_iter: int = 40, eps: float = 0.5, seed: int = 0):
    """omni_kmeans_lab_batch: frames [F, H, W, 3] BGR u8 -> (centres float32 [F, K, 3], compactness float64 [F]), every frame
    clustered on its own with the shared sample indices (None: every pixel)."""
    frames = np.asarray(frames)
    npix = frames.shape[1] * frames.shape[2]
    n = npix if sample_idx is None else len(sample_idx)
    _check(n, npix, sample_idx, K, attempts, max_iter, eps)
    ctrs = np.empty((frames.shape[0], K, 3), np.float32)
    comps = np.empty(frames.shape[0], np.float64)
    for f in range(frames.shape[0]):
        s = lab_samples(frames[f:f + 1], sample_idx)[0]
        ctrs[f], comps[f] = kmeans_frame(s, K, attempts, max_iter, eps, seed)
    return ctrs, comps


def kmeans_lab(img, K: int, sample_idx=None, attempts: int = 3, max_iter: int = 40, eps: float = 0.5, seed: int = 0):
    """omni_kmeans_lab: img [H, W, 3] BGR u8 (any strides) -> (centres float32 [K, 3], compactness)."""
    ctr, comp = kmeans_lab_batch(np.asarray(img)[None], K, sample_idx, attempts, max_iter, eps, seed)
    return ctr[0], float(comp[0])
