"""CPU: the drop-in boundary artefacts (SURVEY.md 8(b)).

* `integration/ape/_C.py` satisfies the reference's import contract (`from ape import _C`,
  ape/layers/multi_scale_deform_attn.py:415-423): with it in place the reference module file defines the real
  MultiScaleDeformableAttention class and finds `torch.ops.ape.ms_deform_attn_forward`.
* every `_target_` override INTEGRATION.md tells a user to pass names a node of the reference's own LazyConfig tree
  (configs/…/ape_deta_vitl_eva02_clip_vlf_lsj1024_cp_16x4_1080k.py and the files it builds on), and the engine class behind
  it accepts every keyword the config passes to the reference class.
* `Instances.to_detectron2()` maps the fields onto detectron2's types.
* entity gates and thing-class slicing of the instance branch (deformable_detr_segm_vl.py:575-593).

What the reference imports and calls, and its config tree (parsed with `ast`: detectron2 is not installed), are recorded in
tests/golden/reference_integration.json by tests/golden/gen_reference_golden.py."""
import importlib
import importlib.util
import inspect
import json
import os
import re
import sys
import types

import pytest
import torch

from conftest import GOLDEN

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _reference():
    with open(os.path.join(GOLDEN, "reference_integration.json")) as f:
        return json.load(f)


def _load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_shipped_C_shim_satisfies_the_reference_import_contract(built):
    ref = _reference()
    assert ref["msda_module_imports_from_ape"] == ["_C"]  # the module's only import from the package: its `try` guard
    assert "ms_deform_attn_forward" in ref["msda_module_ops"]
    saved = {k: sys.modules.get(k) for k in ("ape", "ape._C")}
    try:
        pkg = types.ModuleType("ape")
        pkg.__path__ = [os.path.join(ROOT, "integration", "ape")]
        sys.modules["ape"] = pkg
        sys.modules.pop("ape._C", None)
        ns = {}
        exec("from ape import _C", ns)  # the statement the reference's module runs; ImportError would select its dummy class
        assert ns["_C"].__file__ == os.path.join(ROOT, "integration", "ape", "_C.py")
        for op in ref["msda_module_ops"]:
            assert hasattr(torch.ops.ape, op), f"the reference calls torch.ops.ape.{op}, which the shim does not register"
        schema = str(torch.ops.ape.ms_deform_attn_forward.default._schema)
        assert "Tensor value, Tensor spatial_shapes, Tensor level_start_index, Tensor sampling_loc, Tensor attn_weight, int im2col_step" in schema
        with pytest.raises(RuntimeError, match="Not implemented on the CPU"):  # ms_deform_attn.h:39
            z = torch.zeros
            torch.ops.ape.ms_deform_attn_forward(z(1, 4, 4, 16), z(1, 2, dtype=torch.long), z(1, dtype=torch.long),
                                                 z(1, 3, 4, 1, 4, 2), z(1, 3, 4, 1, 4), 64)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_integration_target_overrides_name_real_config_nodes(built):
    tree = _reference()["model_tree"]
    assert tree["_target_"] == "SomeThing" and tree["model_vision"]["_target_"] == "DeformableDETRSegmVL"
    text = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    overrides = re.findall(r"(model(?:\.\w+)+)\._target_=(ape_b200(?:\.\w+)+)", text)
    assert len(overrides) >= 9
    import ape_b200  # noqa: F401
    for path, target in overrides:
        node = tree
        for k in path.split(".")[1:]:
            assert isinstance(node, dict) and k in node, f"INTEGRATION.md overrides {path}: `{k}` is not a key of the reference config"
            node = node[k]
        assert isinstance(node, dict) and "_target_" in node, f"{path} is not a LazyCall node in the reference config"
        mod, cls = target.rsplit(".", 1)
        engine_cls = getattr(importlib.import_module(mod), cls)
        assert engine_cls.__name__ == node["_target_"], f"{path}: reference builds {node['_target_']}, override names {cls}"
        params = inspect.signature(engine_cls.__init__).parameters
        accepts_kwargs = any(p.kind == p.VAR_KEYWORD for p in params.values())
        for kw in node:
            if kw != "_target_":
                assert accepts_kwargs or kw in params, f"{target} does not accept the config keyword `{kw}` of {path}"


def test_instances_to_detectron2_maps_fields(monkeypatch):
    from ape_b200.structures import Boxes, Instances

    class D2Boxes:
        def __init__(self, tensor):
            self.tensor = tensor

    class D2Instances:
        def __init__(self, image_size, **kw):
            self.image_size = image_size
            self.fields = {}
            for k, v in kw.items():
                self.set(k, v)

        def set(self, k, v):
            self.fields[k] = v

        def __setattr__(self, k, v):
            if k in ("image_size", "fields"):
                object.__setattr__(self, k, v)
            else:
                self.fields[k] = v

    d2 = types.ModuleType("detectron2")
    d2s = types.ModuleType("detectron2.structures")
    d2s.Boxes, d2s.Instances = D2Boxes, D2Instances
    monkeypatch.setitem(sys.modules, "detectron2", d2)
    monkeypatch.setitem(sys.modules, "detectron2.structures", d2s)
    inst = Instances((48, 64), pred_boxes=Boxes(torch.rand(3, 4)), scores=torch.rand(3), pred_classes=torch.arange(3))
    out = inst.to_detectron2()
    assert isinstance(out, D2Instances) and out.image_size == (48, 64)
    assert isinstance(out.fields["pred_boxes"], D2Boxes) and torch.equal(out.fields["pred_boxes"].tensor, inst.pred_boxes.tensor)
    assert torch.equal(out.fields["scores"], inst.scores) and torch.equal(out.fields["pred_classes"], inst.pred_classes)


def test_entity_gates_and_thing_class_slicing(built):
    """deformable_detr_segm_vl.py:575-593 / :628-630 / :671-673 and deformable_detr.py:246-262, 524-532."""
    from ape_b200 import configs
    from ape_b200.modeling import build_model

    m = build_model(configs.MINI)
    name = m.dataset_names[0]
    box_cls = torch.randn(1, 5, 12)
    assert m._detector_box_cls(box_cls) is box_cls          # no dataset selected (eval_dataset_id = -1): all classes
    things, stuff = [f"t{i}" for i in range(8)], [f"s{i}" for i in range(4)]
    m.dataset_stuff = {name: (things, stuff)}
    m.set_eval_dataset(name)
    assert m.eval_dataset_entity == "thing+stuff"
    assert torch.equal(m._detector_box_cls(box_cls), box_cls[..., :8])   # disjoint lists: the first len(things) columns
    m.dataset_stuff = {name: (things[:4], things, None, [0, 2, 5, 7])}   # thing classes are a subset of the stuff classes
    m.set_eval_dataset(name)
    out = m._detector_box_cls(box_cls)
    assert torch.equal(out[..., [0, 2, 5, 7]], box_cls[..., [0, 2, 5, 7]]) and torch.isinf(out[..., [1, 3, 4, 6, 8]]).all()
    m.dataset_stuff = {name: ([], stuff)}
    m.set_eval_dataset(name)
    assert m.eval_dataset_entity == "stuff"                  # instance branch is skipped for stuff-only datasets
    m.set_eval_dataset("some_other_dataset")
    assert m.eval_dataset_id == -1 and m.eval_dataset_entity == ""
