"""The reference's stage structure:
  * oracle/refstages.py -- the as-shipped CPU baseline bench.py times on the GPU box -- writes the same files as the unmodified
    reference's `pipeline.py --start-step 1 --end-step 3` wrote for the golden pipeline cases (tools/make_golden.py);
  * the drop-in stage scripts copied beside a copy of the reference's pipeline.py are the files its build_steps()/module_path()
    resolve (INTEGRATION.md, section A), and its own `missing_for_step` bookkeeping accepts the outputs they are expected to write.
    This one imports the reference's runner and runs only when OMNI_REFERENCE_DIR names it."""
import importlib.util
import json
import os
import shutil
import subprocess
import sys

import cv2
import numpy as np
import pytest

from conftest import REFERENCE_DIR as REF
from helpers import PIPE_CASES, load_pipe_case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DROPIN = os.path.join(ROOT, "omnirevolve-image-processor_b200", "image_processor")


def _files(outdir, names):
    return (cv2.imread(os.path.join(outdir, "resized.png"), cv2.IMREAD_COLOR),
            [cv2.imread(os.path.join(outdir, n, "mask.png"), cv2.IMREAD_GRAYSCALE) for n in names],
            [cv2.imread(os.path.join(outdir, n, "edges.png"), cv2.IMREAD_GRAYSCALE) for n in names],
            cv2.imread(os.path.join(outdir, "edges_composite.png"), cv2.IMREAD_COLOR),
            json.load(open(os.path.join(outdir, "palette_by_name.json"))))


def test_refstages_equals_reference_pipeline(tmp_path):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    for case in PIPE_CASES:
        z, meta = load_pipe_case(case)
        src = tmp_path / f"{case}.png"
        cv2.imwrite(str(src), z["input"])
        out_port = tmp_path / case
        out_port.mkdir()
        cfg = dict(meta["config"], input_image=str(src), output_dir=str(out_port))
        (out_port / "config.json").write_text(json.dumps(cfg))
        for st in ("01", "02", "03"):
            r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "refstages.py"), st],
                               env=dict(env, CONFIG_PATH=str(out_port / "config.json")), stdout=subprocess.PIPE,
                               stderr=subprocess.STDOUT, text=True)
            assert r.returncode == 0, r.stdout[-2000:]
        resized, masks, edges, comp, palette = _files(str(out_port), meta["names"])
        assert np.array_equal(resized, z["resized"]), case
        for i, n in enumerate(meta["names"]):
            assert np.array_equal(masks[i], z["masks"][i]) and np.array_equal(edges[i], z["edges"][i]), (case, n)
        assert np.array_equal(comp, z["composite"]) and palette == meta["palette_by_name"], case


@pytest.mark.reference
def test_reference_pipeline_resolves_the_dropins(tmp_path):
    """Copy the reference's runner + config module and OUR stage scripts into one directory, as INTEGRATION.md A says, and ask
    the runner itself which files it would launch and which outputs it waits for."""
    d = tmp_path / "image_processor"
    d.mkdir()
    for f in ("pipeline.py", "config.py"):
        shutil.copy(os.path.join(REF, f), d / f)
    for f in os.listdir(DROPIN):
        if f.endswith(".py") and f != "config.py":
            shutil.copy(os.path.join(DROPIN, f), d / f)
    sys.path.insert(0, str(d))
    try:
        spec = importlib.util.spec_from_file_location("ref_pipeline_copy", str(d / "pipeline.py"))
        pl = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(pl)
        steps = pl.build_steps()                                    # [(title, path)] (pipeline.py:66-82)
        for i, script in enumerate(("01_resize.py", "02_color_extract.py", "03_edge_detect.py")):
            assert os.path.samefile(steps[i][1], d / script)        # the runner launches OUR file
            assert os.path.samefile(pl.module_path(script), d / script)
            assert "omni_b200" in open(steps[i][1]).read()
        # the runner's resume bookkeeping names exactly the files our stages write (pipeline.py:113-145)
        out = tmp_path / "out"
        names = ["layer_dark", "layer_mid"]
        need = pl.missing_for_step(4, str(out), names)
        assert set(need) == {str(out / "resized.png")} | {str(out / n / f) for n in names for f in ("mask.png", "edges.png")}
    finally:
        sys.path.remove(str(d))
        sys.modules.pop("config", None)
