"""Import the UNMODIFIED reference (upstream stevenczwu/SAMBLE) from the checkout
named by the SAMBLE_REFERENCE environment variable.

Used by make_golden.py and by the `needs_reference` tests that pin the oracle
against the real thing. The repository does not ship the reference: without
SAMBLE_REFERENCE those tests skip, and the committed golden vectors
(tests/test_oracle_golden.py) keep the oracle pinned to the reference's outputs.

The reference is driven by hydra/OmegaConf (train_shapenet.py:27,41-43); neither
is installed, so the YAML trees are read with PyYAML and merged with the same
"dicts merge, leaves replace" rule. The `wandb` subtree (default.yaml holds a
third-party API key there) is dropped on load and never written anywhere.
"""
from __future__ import annotations

import copy
import os
import sys

REF_ROOT = os.environ.get("SAMBLE_REFERENCE", "")


def available() -> bool:
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "utils", "ops.py"))


def _yaml(name: str) -> dict:
    import yaml

    with open(os.path.join(REF_ROOT, "configs", name)) as f:
        tree = yaml.safe_load(f)
    tree.pop("wandb", None)
    return tree


def reference_config(which: str, **overrides):
    """default.yaml (+) seg.yaml|cls.yaml as a samble_b200.config.Cfg."""
    from samble_b200.config import Cfg

    cfg = Cfg(_yaml("default.yaml")).merged(_yaml(f"{which}.yaml"))
    flb = cfg.feature_learning_block
    for k, v in overrides.items():
        node = flb
        parts = k.split(".")
        for p in parts[:-1]:
            node = node[p]
        node[parts[-1]] = v
    return cfg


def modules():
    """(ops, embedding, attention, downsample, upsample, seg_model, cls_model) of the reference."""
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    from utils import ops  # noqa
    from models import attention, cls_model, downsample, embedding, seg_model, upsample  # noqa

    return ops, embedding, attention, downsample, upsample, seg_model, cls_model


def build_model(which: str, cfg):
    """Reference model from a config; deep-copied because DownSampleToken.__init__
    mutates the bin_boundaries list in place (models/downsample.py:98-99)."""
    _, _, _, _, _, seg_model, cls_model = modules()
    cfg = copy.deepcopy(cfg)
    if which == "seg":
        return seg_model.ShapeNetModel(cfg)
    return cls_model.ModelNetModel(cfg)
