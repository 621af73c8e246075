"""oracle/kmeans_model.py, the NumPy restatement of the device k-means that tests/test_gpu_kmeans_exact.py holds the kernel to bit
for bit.  These tests check the model itself, without a GPU: its quality against cv2.kmeans, its own compactness figure, its
determinism, degenerate inputs, and its vectorised steps against a loop-by-loop transliteration of kmeans.cu on small inputs."""
import cv2
import numpy as np
import pytest

from helpers import KMEANS_TOL, compactness, lab_sample, synth, uniform_img
from oracle import cmodel
from oracle import kmeans_model as km

CRIT = (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_MAX_ITER, 40, 0.5)


def _bound(n, exact):
    """The model's compactness is a sum of float32 distances rounded to 1/1024: at most half a unit per sample, plus the float32
    rounding of each distance."""
    return n * 0.5 / 1024 + 1e-6 * exact


@pytest.mark.parametrize("K", [2, 4, 8, 16])
@pytest.mark.parametrize("shape,seed", [((600, 800), 1), ((480, 480), 2)])
def test_quality_within_tolerance_of_cv2(K, shape, seed):
    img = synth(shape[0], shape[1], seed)
    idx, lab = lab_sample(img)
    cv2.setRNGSeed(0)
    comp_cv, _l, _c = cv2.kmeans(lab, K, None, CRIT, 3, cv2.KMEANS_PP_CENTERS)
    ctr, comp = km.kmeans_lab(img, K, idx)
    mine = compactness(lab, ctr)
    assert mine <= (1.0 + KMEANS_TOL) * comp_cv, (K, mine / comp_cv)
    assert abs(comp - mine) <= _bound(len(lab), mine)


@pytest.mark.parametrize("K,attempts,max_iter,eps", [(1, 1, 40, 0.5), (3, 2, 1, 0.5), (8, 3, 40, 0.0), (32, 1, 5, 0.5)])
def test_compactness_is_the_float64_figure_of_the_centres(K, attempts, max_iter, eps):
    img = uniform_img(90, 110, K)
    lab = cmodel.bgr2lab(img).reshape(-1, 3).astype(np.float64)
    ctr, comp = km.kmeans_lab(img, K, None, attempts, max_iter, eps, seed=K)
    mine = compactness(lab, ctr)
    assert abs(comp - mine) <= _bound(len(lab), mine)
    assert comp * 1024 == int(comp * 1024)                              # a whole number of 1/1024 units


def test_deterministic_and_seeded():
    img = synth(200, 300, 4)
    idx = np.random.default_rng(1).choice(200 * 300, 20_000, replace=False)
    a = km.kmeans_lab(img, 8, idx, seed=3)
    b = km.kmeans_lab(img, 8, idx, seed=3)
    assert np.array_equal(a[0], b[0]) and a[1] == b[1]
    c = km.kmeans_lab(img, 8, idx, seed=4)
    assert not np.array_equal(a[0], c[0])


def test_flat_image():
    img = np.full((40, 60, 3), (30, 160, 90), np.uint8)
    lab = cmodel.bgr2lab(img[:1, :1]).reshape(3).astype(np.float32)
    ctr, comp = km.kmeans_lab(img, 4)
    assert comp == 0.0 and (ctr == lab).all()


def test_two_colours_eight_centres():
    cols = np.array([[20, 20, 200], [240, 200, 10]], np.uint8)
    img = cols[np.random.default_rng(0).integers(0, 2, (50, 41))]
    lab = cmodel.bgr2lab(cols[None])[0].astype(np.float32)
    ctr, comp = km.kmeans_lab(img, 8)
    assert comp == 0.0
    assert {tuple(c) for c in ctr} == {tuple(c) for c in lab}            # duplicate centres; empty clusters keep theirs


def test_as_many_samples_as_centres():
    img = uniform_img(1, 9, 5)
    lab = cmodel.bgr2lab(img)[0].astype(np.float32)
    ctr, comp = km.kmeans_lab(img, 9)
    assert comp == 0.0
    assert sorted(map(tuple, ctr)) == sorted(map(tuple, lab))


def test_one_centre_is_the_mean():
    img = synth(70, 90, 8)
    s = cmodel.bgr2lab(img).reshape(-1, 3).astype(np.float64)
    ctr, comp = km.kmeans_lab(img, 1)
    assert np.array_equal(ctr[0], (s.sum(axis=0) / len(s)).astype(np.float32))
    assert abs(comp - compactness(s, ctr)) <= _bound(len(s), comp)


def test_outside_the_kernel_domain_is_refused():
    img = uniform_img(2, 2, 0)
    for kw in (dict(K=5), dict(K=2, attempts=65), dict(K=2, max_iter=0), dict(K=2, eps=-1.0), dict(K=33)):
        with pytest.raises(ValueError):
            km.kmeans_lab(img, **kw)


# ---- the vectorised model against kmeans.cu transliterated loop by loop ---------------------------------------------------------
f32 = np.float32


def _d2(s, c):
    d = [f32(f32(s[q]) - c[q]) for q in range(3)]
    return f32(f32(f32(d[0] * d[0]) + f32(d[1] * d[1])) + f32(d[2] * d[2]))


def _loop_run(s, K, seed, attempt, max_iter, eps):
    """One run of fk_km_seed, fk_km_assign / fk_km_update and the forced assignment, one sample at a time."""
    n, per = len(s), (len(s) + 1023) // 1024
    ctr = [[f32(v) for v in s[min(n - 1, int(km.km_uniform(seed, attempt, 0, 0) * n))]]]
    dist = [_d2(p, ctr[0]) for p in s]

    def thread_sums():
        return [float(sum(dist[min(n, t * per):min(n, t * per + per)])) for t in range(1024)]
    s_thr = thread_sums()
    for k in range(1, K):
        total, picks = sum(s_thr), []
        for t in range(3):
            r = km.km_uniform(seed, attempt, k, t + 1) * total
            acc, th = 0.0, 1023
            for i in range(1024):
                if acc + s_thr[i] > r:
                    th = i
                    break
                acc += s_thr[i]
            a = min(n, th * per)
            b = min(n, a + per)
            pick = max(a, b - 1)
            for i in range(a, b):
                acc += float(dist[i])
                if acc > r:
                    pick = i
                    break
            picks.append(min(max(pick, 0), n - 1))
        pots = [sum(float(min(dist[i], _d2(s[i], [f32(v) for v in s[p]]))) for i in range(n)) for p in picks]
        bt = 0
        for t in (1, 2):
            if pots[t] < pots[bt]:
                bt = t
        ctr.append([f32(v) for v in s[picks[bt]]])
        dist = [min(dist[i], _d2(s[i], ctr[k])) for i in range(n)]
        s_thr = thread_sums()

    def assign():
        sums, comp = [[0] * 4 for _ in range(K)], 0
        for p in s:
            bd, best = f32(3.0e38), 0
            for k in range(K):
                d = _d2(p, ctr[k])
                if d < bd:
                    bd, best = d, k
            for q in range(3):
                sums[best][q] += int(p[q])
            sums[best][3] += 1
            comp += int(f32(f32(bd * f32(1024)) + f32(0.5)))
        return sums, comp
    eps2 = f32(f32(eps) * f32(eps))
    for _ in range(max_iter):
        sums, _c = assign()
        shift = f32(0)
        for k in range(K):
            if sums[k][3]:
                d2 = f32(0)
                for q in range(3):
                    c = f32(sums[k][q] / sums[k][3])
                    d2 = f32(d2 + f32(f32(c - ctr[k][q]) * f32(c - ctr[k][q])))
                    ctr[k][q] = c
                shift = max(shift, d2)
        if shift <= eps2:
            break
    return np.array(ctr, np.float32), assign()[1]


def _loop_kmeans(s, K, attempts, max_iter, eps, seed):
    runs = [_loop_run(s, K, seed, a, max_iter, eps) for a in range(attempts)]
    best = min(range(attempts), key=lambda a: (runs[a][1], a))
    return runs[best][0], runs[best][1] / 1024.0


def _grey(levels, n, seed):
    """Lab samples on the grey axis with L = levels: ties in the assignment (half-integer centres) and in the seeding."""
    return np.array([[v, 128, 128] for v in levels], np.int32)[np.random.default_rng(seed).integers(0, len(levels), n)]


@pytest.mark.parametrize("case", ["noise", "few_iters_eps0", "flat_above_1024", "two_colours", "n_eq_K", "grey_ties", "big_seed"])
def test_vectorised_model_equals_the_loops(case):
    rng = np.random.default_rng(7)
    s, K, attempts, max_iter, eps, seed = {
        "noise": (rng.integers(0, 256, (300, 3)), 5, 3, 40, 0.5, 0),
        "few_iters_eps0": (rng.integers(0, 256, (2500, 3)), 3, 2, 3, 0.0, 9),
        "flat_above_1024": (np.full((1500, 3), 77), 4, 2, 5, 0.5, 3),
        "two_colours": (np.array([[10, 128, 128], [200, 100, 150]])[rng.integers(0, 2, 2100)], 8, 3, 5, 0.5, 7),
        "n_eq_K": (rng.integers(0, 256, (6, 3)), 6, 3, 40, 0.5, 2),
        "grey_ties": (_grey(range(108, 114), 400, 1), 3, 3, 40, 0.5, 5),
        "big_seed": (rng.integers(0, 256, (200, 3)), 4, 2, 40, 0.5, 2 ** 64 - 1),
    }[case]
    s = np.asarray(s, np.int32)
    want = _loop_kmeans(s, K, attempts, max_iter, eps, seed)
    got = km.kmeans_frame(s, K, attempts, max_iter, eps, seed)
    assert np.array_equal(got[0].view(np.uint32), want[0].view(np.uint32)) and got[1] == want[1]
