"""stages.frame_centers(mode="host"): every frame's centres are those of a fresh-process stage-02 run on that frame, whether the
frames run one after another or on threads (OpenCV's RNG is per thread).  CPU only: cv2.kmeans and NumPy."""
import json
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np

from helpers import synth, uniform_img

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "omnirevolve-image-processor_b200")


def _fresh_process_centers(path, k):
    """kmeans_lab_centers on one frame in a new interpreter: the process-global RNG state a stage-02 run starts from."""
    code = ("import sys, json, numpy as np; sys.path.insert(0, %r); from omni_b200 import stages; "
            "img = np.load(%r); print(json.dumps(stages.kmeans_lab_centers(img, %d).tolist()))" % (PKG, str(path), k))
    env = {kk: v for kk, v in os.environ.items() if kk != "OMNI_B200_KMEANS"}
    r = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    return np.array(json.loads(r.stdout.strip().splitlines()[-1]), np.float32)


def test_host_mode_equals_fresh_process_runs(tmp_path, monkeypatch):
    monkeypatch.delenv("OMNI_B200_KMEANS", raising=False)
    from omni_b200 import stages
    # 520 x 400 = 208k pixels: above the 200k sample limit, so the seeded subsample is drawn as in the reference
    frames = np.stack([synth(520, 400, 11), uniform_img(520, 400, 12), synth(520, 400, 13, cell=8)])
    cfg = SimpleNamespace(color_names=["layer_dark", "layer_mid", "layer_skin", "layer_light", "x5", "x6"])
    K = 6
    want = []
    for i, f in enumerate(frames):
        np.save(tmp_path / f"f{i}.npy", f)
        want.append(_fresh_process_centers(tmp_path / f"f{i}.npy", K))
    want = np.stack(want)
    serial, luts = stages.frame_centers(frames, cfg, mode="host", threads=1)
    threaded, luts_t = stages.frame_centers(frames, cfg, mode="host", threads=3)
    assert serial.shape == (3, K, 3) and serial.dtype == np.float32 and luts.shape == (3, K) and luts.dtype == np.uint8
    assert np.array_equal(serial, want)
    assert np.array_equal(threaded, want) and np.array_equal(luts_t, luts)
    for c, lut in zip(want, luts):
        assert np.array_equal(lut, stages.darkness_lut(c)[1])
    # frames that are not one array (images of different sizes) work in host mode too
    mixed, _ = stages.frame_centers([frames[0], frames[1][:300]], cfg, mode="host", threads=2)
    assert np.array_equal(mixed[0], want[0]) and mixed.shape == (2, K, 3)


def test_k_and_sample_settings_follow_stage02():
    from omni_b200 import stages
    cfg = SimpleNamespace(color_names=["a", "b", "c", "d"], cluster_k=9, kmeans_sample_limit=5000, kmeans_attempts=2)
    assert stages._kmeans_args(cfg) == (4, 5000, 2)
    cfg = SimpleNamespace(color_names=["a"])
    assert stages._kmeans_args(cfg)[0] == 2
    c, l = stages.frame_centers(np.zeros((0, 8, 8, 3), np.uint8), cfg)
    assert c.shape == (0, 2, 3) and l.shape == (0, 2)
