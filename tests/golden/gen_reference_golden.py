"""Generates the fixtures that let the CPU tests compare against the reference without its sources at hand:

* reference_integration.json  what the reference imports from `ape` and which `torch.ops.ape` operators it calls in
                              ape/layers/multi_scale_deform_attn.py, and the model tree of its LazyConfig files
                              (configs/…/ape_deta_vitl_eva02_clip_vlf_lsj1024_cp_16x4_1080k.py and the files it builds on),
                              parsed with `ast` (detectron2 is not installed) — tests/test_integration_cpu.py
* state_dict_reference.npz    names and shapes of the reference model's state_dict per spec — tests/test_state_dict_cpu.py
* vlf_reference.npz           the reference BiAttentionBlock (ape/layers/fuse_helper.py) on seeded inputs with the synthetic
                              weights, a seeded sample of vision rows and every language row — tests/test_vlf_cpu.py
* panoptic_reference.npz      the reference's DeformableDETRSegmVL._postprocess_panoptic on the seeded predictions of
                              tests/test_panoptic_cpu.py

Needs a checkout of the reference (its directory in APE_REFERENCE, see oracle/refshim.py) and a built ape_b200:
    python tests/golden/gen_reference_golden.py"""
import ast
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from oracle import refshim  # noqa: E402

REF = refshim.REF

# ---- LazyConfig tree from the config sources -----------------------------------------------------------------------
LEAF = "<value>"


def _lazy_tree(node, env):
    """`L(Target)(kw=...)` -> {"_target_": "Target", kw: subtree | LEAF}; a bare name bound to a tree -> that tree."""
    if isinstance(node, ast.Call) and isinstance(node.func, ast.Call) and getattr(node.func.func, "id", "") == "L":
        tgt = node.func.args[0]
        name = tgt.id if isinstance(tgt, ast.Name) else ast.unparse(tgt)
        return {"_target_": name, **{kw.arg: _lazy_tree(kw.value, env) for kw in node.keywords if kw.arg}}
    if isinstance(node, ast.Name) and isinstance(env.get(node.id), dict):
        return env[node.id]
    return LEAF


def _attr_path(t):
    path = []
    while isinstance(t, ast.Attribute):
        path.append(t.attr)
        t = t.value
    return (t.id if isinstance(t, ast.Name) else None), path[::-1]


def _run_config(src, env):
    """The three statement forms the configs use to build the model tree: `name = L(..)(..)`,
    `name.a.b = <L-call | value>` and `name.a.b.update(_target_=X, ...)`."""
    for stmt in ast.parse(src).body:
        if isinstance(stmt, ast.Assign) and len(stmt.targets) == 1:
            tgt = stmt.targets[0]
            if isinstance(tgt, ast.Name):
                tree = _lazy_tree(stmt.value, env)
                if isinstance(tree, dict):
                    env[tgt.id] = tree
                continue
            root, path = _attr_path(tgt)
            node = env.get(root)
            for k in path[:-1]:
                node = node.get(k) if isinstance(node, dict) else None
            if isinstance(node, dict) and path:
                node[path[-1]] = _lazy_tree(stmt.value, env)
        elif isinstance(stmt, ast.Expr) and isinstance(stmt.value, ast.Call) and isinstance(stmt.value.func, ast.Attribute) \
                and stmt.value.func.attr == "update":
            root, path = _attr_path(stmt.value.func.value)
            node = env.get(root)
            for k in path:
                node = node.get(k) if isinstance(node, dict) else None
            if isinstance(node, dict):
                for kw in stmt.value.keywords:
                    if kw.arg == "_target_":
                        node["_target_"] = kw.value.id if isinstance(kw.value, ast.Name) else ast.unparse(kw.value)
                    elif kw.arg:
                        node[kw.arg] = _lazy_tree(kw.value, env)


def reference_model_tree():
    env = {}
    for rel in ("configs/common/backbone/vitl_eva02_clip.py",
                "configs/COCO_InstanceSegmentation/ape_deta/models/ape_deta_r50.py",
                "configs/LVISCOCOCOCOSTUFF_O365_OID_VGR_SA1B_REFCOCO_GQA_PhraseCut_Flickr30k/ape_deta/"
                "ape_deta_vitl_eva02_clip_vlf_lsj1024_cp_16x4_1080k.py"):
        _run_config(open(os.path.join(REF, rel)).read(), env)
    tree = env["model"]
    assert tree["_target_"] == "SomeThing" and tree["model_vision"]["_target_"] == "DeformableDETRSegmVL"
    return tree


def msda_import_contract():
    """Names the MSDA module imports from the `ape` package and the `torch.ops.ape` operators it calls."""
    src = open(os.path.join(REF, "ape", "layers", "multi_scale_deform_attn.py")).read()
    imports, ops = set(), set()
    for node in ast.walk(ast.parse(src)):
        if isinstance(node, ast.ImportFrom) and node.module == "ape":
            imports.update(a.name for a in node.names)
        if isinstance(node, ast.Attribute) and ast.unparse(node.value) == "torch.ops.ape":
            ops.add(node.attr)
    return sorted(imports), sorted(ops)


def gen_integration():
    imports, ops = msda_import_contract()
    out = {"msda_module_imports_from_ape": imports, "msda_module_ops": ops, "model_tree": reference_model_tree()}
    with open(os.path.join(HERE, "reference_integration.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
        f.write("\n")
    print("integration", imports, ops)


def gen_state_dict():
    from ape_b200 import configs
    from oracle import ref_model
    from test_state_dict_cpu import SPECS

    arrays = {}
    for name in SPECS:
        ref, _ = ref_model.build_reference_model(getattr(configs, name), num_text=16)
        sd = ref.state_dict()
        arrays[f"{name}.names"] = np.array(list(sd))
        arrays[f"{name}.shapes"] = np.array([",".join(map(str, v.shape)) for v in sd.values()])
        print("state_dict", name, len(sd))
    np.savez_compressed(os.path.join(HERE, "state_dict_reference.npz"), **arrays)


def gen_vlf():
    from test_vlf_cpu import reference_case

    refshim.install()
    fh = refshim.load("ape.layers.fuse_helper")
    ref = fh.BiAttentionBlock(v_dim=256, l_dim=128, embed_dim=512, num_heads=8, dropout=0.0, drop_path=0.0, init_values=1 / 6,
                              stable_softmax_2d=True, clamp_min_for_underflow=True, clamp_max_for_overflow=True).eval()
    mine, v, l, rows = reference_case()
    ref.load_state_dict(mine.state_dict())
    with torch.no_grad():
        rv, rl = ref(v, l, attention_mask_v=None, attention_mask_l=None)
    np.savez_compressed(os.path.join(HERE, "vlf_reference.npz"), v_rows=rv[:, rows].numpy(), l=rl.numpy())
    print("vlf", tuple(rv.shape), tuple(rl.shape))


def gen_panoptic():
    from test_panoptic_cpu import CASES, panoptic_case

    refshim.install()
    segm = refshim.load("ape.modeling.ape_deta.deformable_detr_segm_vl")
    arrays = {}
    for seed, K, n_cls, stuff_first in CASES:
        mask_cls, mask_pred, image_size, out_hw, meta, cfg, images = panoptic_case(seed, K, n_cls, stuff_first)
        seg, info = segm.DeformableDETRSegmVL._postprocess_panoptic([mask_cls], [mask_pred],
                                                                   [{"height": out_hw[0], "width": out_hw[1]}],
                                                                   images, meta, cfg)[0]["panoptic_seg"]
        arrays[f"seg{seed}"] = seg.numpy()
        arrays[f"info{seed}"] = np.array(json.dumps(info))
        print("panoptic", seed, len(info))
    np.savez_compressed(os.path.join(HERE, "panoptic_reference.npz"), **arrays)


if __name__ == "__main__":
    assert refshim.available(), f"no reference checkout at {REF}: set APE_REFERENCE"
    gen_integration()
    gen_state_dict()
    gen_vlf()
    gen_panoptic()
