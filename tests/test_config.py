import copy
import glob
import os

import pytest
import yaml

from msrflute_b200.core.config import ConfigNode, FLUTEConfig
from msrflute_b200.core.schema import SCHEMA
from msrflute_b200.core.validator import Validator

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# The configs shipped by the original FLUTE (microsoft/msrflute @ 8bfe0854), same layout: they must keep validating.
REF_CONFIGS = os.path.join(ROOT, "tests", "golden", "reference_configs")


def _yamls():
    pats = []
    for base in (ROOT, REF_CONFIGS):
        pats += [os.path.join(base, "experiments", "*", "config.yaml"), os.path.join(base, "configs", "*.yaml"),
                 os.path.join(base, "testing", "*.yaml")]
    out = []
    for p in pats:
        out += sorted(glob.glob(p))
    return out


@pytest.mark.parametrize("path", _yamls())
def test_schema_accepts_every_shipped_yaml(path):
    with open(path) as f:
        raw = yaml.safe_load(f)
    cfg = FLUTEConfig.from_dict(raw)
    assert cfg["server_config"]["val_freq"] >= 1
    # defaults of schema.py:106-111,123-134 are filled in
    assert cfg["client_config"]["data_config"]["train"]["max_grad_norm"] == raw["client_config"]["data_config"]["train"].get("max_grad_norm", 5.0)
    assert cfg["server_config"]["data_config"]["val"]["num_workers"] >= 0


def _minimal():
    with open(os.path.join(ROOT, "experiments", "cv_lr_mnist", "config.yaml")) as f:
        return yaml.safe_load(f)


def test_missing_required_key_is_reported():
    raw = _minimal()
    del raw["server_config"]["softmax_beta"]
    with pytest.raises(ValueError, match="softmax_beta"):
        FLUTEConfig.from_dict(raw)


def test_forbidden_num_clients_and_bad_enum():
    raw = _minimal()
    raw["server_config"]["data_config"]["num_clients"] = 5
    with pytest.raises(ValueError):
        FLUTEConfig.from_dict(raw)
    raw = _minimal()
    raw["server_config"]["optimizer_config"]["type"] = "rmsprop"
    with pytest.raises(ValueError):
        FLUTEConfig.from_dict(raw)


def test_cerberus_strict_float_vs_lenient():
    v = Validator(SCHEMA, allow_unknown=True, lenient_numbers=False)
    raw = _minimal()
    raw["server_config"]["optimizer_config"]["lr"] = 1          # int where float is required
    assert not v.validate(raw)
    assert Validator(SCHEMA, allow_unknown=True, lenient_numbers=True).validate(raw)


def test_config_node_semantics():
    c = ConfigNode({"a": {"b": {"c": 3}}, "n": None})
    assert c["a"]["b"]["c"] == 3 and c.a.b.c == 3
    assert c.lookup("a.b.c") == 3 and c.lookup("a.x.c", 7) == 7
    assert "n" not in c and c.get("n", 5) == 5           # None counts as absent (reference Config semantics)
    assert c.pop("a")["b"]["c"] == 3 and "a" not in c
    d = copy.deepcopy(ConfigNode({"x": [1, 2], "y": {"z": 1}}))
    assert isinstance(d["y"], ConfigNode) and d.to_dict() == {"x": [1, 2], "y": {"z": 1}}


def test_num_clients_per_iteration_string_range():
    raw = _minimal()
    raw["server_config"]["num_clients_per_iteration"] = "3,6"
    assert FLUTEConfig.from_dict(raw)["server_config"]["num_clients_per_iteration"] == "3,6"
