"""The config.json contract: omni_b200.config must expose the reference's keys, defaults and load semantics."""
import dataclasses
import json
import os

from conftest import GOLDEN
from omni_b200 import config as mine


def test_defaults_and_unknown_keys(tmp_path, monkeypatch):
    cfg = mine.Config()
    assert cfg.max_dimension == 2000 and cfg.edge_low_threshold == 50 and cfg.edge_high_threshold == 150
    assert cfg.color_names == ["layer_dark", "layer_mid", "layer_skin", "layer_light"] and cfg.n_cores == 12
    p = tmp_path / "config.json"
    p.write_text(json.dumps({"max_dimension": 512, "extraction_mode": "swatch", "color_names": ["a", "b"], "bogus": 1}))
    monkeypatch.setenv("CONFIG_PATH", str(p))
    c2 = mine.load_config()
    assert c2.max_dimension == 512 and c2.color_names == ["a", "b"]
    assert not hasattr(c2, "extraction_mode") and not hasattr(c2, "bogus")      # unknown keys are dropped (config.py:124-125)
    assert c2._raw["extraction_mode"] == "swatch"
    c2.output_dir = str(tmp_path / "out")
    c2.ensure_output_dirs()
    assert os.path.isdir(tmp_path / "out" / "a") and os.path.isdir(tmp_path / "out" / "b")
    # broken JSON -> defaults, like the reference
    p.write_text("{not json")
    assert mine.load_config().max_dimension == 2000
    # two Config() instances must not share list defaults
    a, b = mine.Config(), mine.Config()
    a.color_names.append("x")
    assert "x" not in b.color_names


def test_same_fields_and_defaults_as_reference():
    """The config.json the unmodified reference's pipeline.py wrote from its dataclass defaults (golden case pipe_default_k4,
    input_image and output_dir dropped when it was frozen): same fields, same order, same defaults."""
    ref = json.load(open(os.path.join(GOLDEN, "pipe_default_k4.json")))["config"]
    mf = [f.name for f in dataclasses.fields(mine.Config)]
    assert mf[:2] == ["input_image", "output_dir"] and mf[2:] == list(ref)
    m0 = mine.Config()
    for name, rv in ref.items():
        assert json.dumps(rv) == json.dumps(getattr(m0, name), default=list), name
