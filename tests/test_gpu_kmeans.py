"""Opt-in device k-means of the Lab centres (omni_kmeans_lab; SURVEY 8f rank 2).  cv2.kmeans cannot be reproduced bit for bit (it
draws from OpenCV's global RNG), so the contract is on the QUALITY of the centres: on the reference's own 200k-pixel subsample the
compactness (sum of squared Lab distances to the nearest centre) is within TOL of what cv2.kmeans reaches with the reference's
criteria, and the call is deterministic.  Needs a B200: `-m gpu`."""
import json
import os
import subprocess
import sys

import cv2
import numpy as np
import pytest

from helpers import KMEANS_TOL as TOL, compactness as _compactness, lab_sample as _sample, synth, uniform_img

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    import omni_b200
    e = omni_b200.Engine(0)
    yield e
    e.close()


@pytest.mark.parametrize("K", [2, 4, 8, 16])
@pytest.mark.parametrize("shape,seed", [((600, 800), 1), ((480, 480), 2)])
def test_compactness_within_tolerance_of_cv2(eng, K, shape, seed):
    img = synth(shape[0], shape[1], seed)
    idx, lab = _sample(img)
    cv2.setRNGSeed(0)
    comp_cv, _l, ctr_cv = cv2.kmeans(lab, K, None, (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_MAX_ITER, 40, 0.5), 3, cv2.KMEANS_PP_CENTERS)
    d = torch.from_numpy(img).cuda()
    ctr, comp = eng.kmeans_lab(d, K, idx)
    assert ctr.shape == (K, 3) and np.isfinite(ctr).all()
    mine = _compactness(lab, ctr)
    assert abs(comp - mine) <= 2e-3 * mine                      # the kernel's own figure (fixed point, float32 distances)
    assert mine <= (1.0 + TOL) * comp_cv, (K, mine / comp_cv)
    ctr2, comp2 = eng.kmeans_lab(d, K, idx)                     # deterministic: integer accumulation, fixed reduction order
    assert np.array_equal(ctr, ctr2) and comp == comp2


def test_every_pixel_mode_and_noise_image(eng):
    img = uniform_img(300, 400, 3)
    _idx, lab = _sample(img)                                    # 120k pixels: below the sample limit
    d = torch.from_numpy(img).cuda()
    ctr, comp = eng.kmeans_lab(d, 8, None, seed=7)
    cv2.setRNGSeed(0)
    comp_cv, _l, _c = cv2.kmeans(lab, 8, None, (cv2.TERM_CRITERIA_EPS + cv2.TERM_CRITERIA_MAX_ITER, 40, 0.5), 3, cv2.KMEANS_PP_CENTERS)
    assert _compactness(lab, ctr) <= (1.0 + TOL) * comp_cv


def test_stage02_with_gpu_kmeans(tmp_path):
    """OMNI_B200_KMEANS=gpu: the drop-in stage 02 takes its centres from the device; the files keep their schema and the masks are
    the exact assignment to the centres written in palette_by_name.json."""
    img = synth(512, 640, 9)
    out = tmp_path / "out"
    out.mkdir()
    cv2.imwrite(str(out / "resized.png"), img)
    names = ["layer_dark", "layer_mid", "layer_skin", "layer_light"]
    cfg = {"input_image": str(out / "resized.png"), "output_dir": str(out), "color_names": names}
    (out / "config.json").write_text(json.dumps(cfg))
    env = dict(os.environ, CONFIG_PATH=str(out / "config.json"), OMNI_B200_KMEANS="gpu", PYTHONUNBUFFERED="1")
    script = os.path.join(ROOT, "omnirevolve-image-processor_b200", "image_processor", "02_color_extract.py")
    r = subprocess.run([sys.executable, script], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:]
    pal = json.load(open(out / "palette_by_name.json"))
    assert sorted(pal) == sorted(names)
    assert sum(pal[n]["pixels"] for n in names) == img.shape[0] * img.shape[1]
    L = [pal[n]["cluster_lab"][0] for n in sorted(names, key=lambda n: pal[n]["cluster_index"])]
    assert L == sorted(L)                                       # dark -> light relabelling as in 02:121-127
    for n in names:
        m = cv2.imread(str(out / n / "mask.png"), cv2.IMREAD_GRAYSCALE)
        assert m.shape == img.shape[:2] and set(np.unique(m)) <= {0, 255} and int((m > 0).sum()) == pal[n]["mask_nonzero"]
