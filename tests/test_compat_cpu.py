"""CPU: the drop-in boundary (SURVEY.md section 8b) -- call signatures equal to the reference's, import-path aliases, and a
checkpoint PICKLED BY THE REFERENCE (tests/golden/ref_tiny.pt, whole-module pickle naming models.yolo.DetectionModel,
models.common.Conv, ...) loading into the engine's classes."""
import inspect
import json
import os
import sys

import numpy as np
import pytest
import torch

from tests.golden.make_golden_cases import SIGNATURE_SURFACE as SURFACE

G = os.path.join(os.path.dirname(__file__), "golden")


def _resolve(mod, qual):
    obj = mod
    for part in qual.split("."):
        obj = getattr(obj, part)
    return obj


def test_signatures_match_the_reference():
    """Every reference parameter (name, position, default) is present in this package's callable; extra trailing keyword
    parameters with defaults are allowed (e.g. non_max_suppression(..., return_indices=False)).  The reference's signatures
    are stored in tests/golden/ref_signatures.json (tests/golden/make_golden.py signatures)."""
    import importlib

    ref = json.load(open(os.path.join(G, "ref_signatures.json")))
    assert sorted(ref) == sorted(f"{mod}:{qual}" for mod, qual in SURFACE)
    bad = []
    for mod, qual in SURFACE:
        ours = inspect.signature(_resolve(importlib.import_module("yolov5_b200." + mod), qual))
        mine = [(n, repr(p.default) if p.default is not inspect._empty else None, str(p.kind)) for n, p in ours.parameters.items()]
        theirs = [tuple(x) for x in ref[f"{mod}:{qual}"]]
        if mine[: len(theirs)] != theirs or any(d is None for _, d, _ in mine[len(theirs):]):
            bad.append((mod, qual, theirs, mine))
    assert not bad, bad


def test_aliases_and_reference_pickled_checkpoint_load():
    from yolov5_b200 import compat
    from yolov5_b200.models.experimental import attempt_load

    try:
        assert compat.install()
        import models.yolo as my
        import utils.general as ug
        from yolov5_b200.models import yolo
        from yolov5_b200.utils import general

        assert my is yolo and ug is general and my.DetectionModel is yolo.DetectionModel
        ck = torch.load(os.path.join(G, "ref_tiny.pt"), map_location="cpu", weights_only=False)
        m = ck["model"]
        assert type(m) is yolo.DetectionModel and type(m.model[0]).__module__ == "yolov5_b200.models.common"
        ref = np.load(os.path.join(G, "ref_tiny_forward.npz"))
        assert list(m.state_dict().keys()) == json.loads(str(ref["keys"]))
        assert m.yaml == json.loads(str(ref["cfg"])) and m.names == {0: "a", 1: "b", 2: "c"} and [float(s) for s in m.stride] == [8.0, 16.0, 32.0]
        # a model built by THIS package from the same cfg has the same parameter set (state_dict interchange both ways)
        twin = yolo.DetectionModel(json.loads(str(ref["cfg"])))
        assert {k: tuple(v.shape) for k, v in twin.state_dict().items()} == {k: tuple(v.shape) for k, v in m.state_dict().items()}
        twin.load_state_dict(m.float().state_dict())
        fused = attempt_load(os.path.join(G, "ref_tiny.pt"), device="cpu")
        assert type(fused) is yolo.DetectionModel and not fused.training and not hasattr(fused.model[0], "bn") and fused.model[0].conv.bias is not None
        import pickle

        pickle.loads(pickle.dumps(fused))  # engine modules stay picklable (train.py:469-482 pickles whole modules)
    finally:
        compat.uninstall()
    assert "models.yolo" not in sys.modules or not sys.modules["models.yolo"].__name__.startswith("yolov5_b200")


def test_forward_accepts_the_reference_keywords():
    from yolov5_b200.models.yolo import DetectionModel

    m = DetectionModel("yolov5n").eval()
    for kw in (dict(augment=False), dict(augment=True), dict(augment=False, profile=False), dict(profile=True)):
        with pytest.raises(RuntimeError, match="CUDA"):  # the call is accepted and reaches the engine, which refuses CPU tensors
            m(torch.zeros(1, 3, 64, 64), **kw)
