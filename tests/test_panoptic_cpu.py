"""CPU: the vectorised panoptic merging (ape_b200/modeling/postprocess.py) against the reference's own
`DeformableDETRSegmVL._postprocess_panoptic` (deformable_detr_segm_vl.py:919-998) — identical segment maps and segments_info
on random predictions.  The reference's results were recorded by tests/golden/gen_reference_golden.py, which executes that
function unmodified under the import shims."""
import json
import os
import types

import numpy as np
import pytest
import torch

from ape_b200.modeling.postprocess import postprocess_panoptic
from conftest import GOLDEN

CASES = [(0, 12, 9, False), (1, 40, 7, True), (2, 3, 5, False), (3, 25, 12, True)]


def panoptic_case(seed, K, n_cls, stuff_first):
    """Seeded predictions and the metadata / config the reference function takes."""
    g = torch.Generator().manual_seed(seed)
    H = W = 48
    image_size, out_hw = (40, 44), (80, 88)
    mask_cls = torch.randn(K, n_cls, generator=g) * 2
    # blobby masks so that queries overlap and compete
    yy, xx = torch.meshgrid(torch.arange(H).float(), torch.arange(W).float(), indexing="ij")
    c = torch.rand(K, 2, generator=g) * 40
    r = torch.rand(K, generator=g) * 12 + 3
    mask_pred = (r[:, None, None] - ((yy[None] - c[:, 0, None, None]) ** 2 + (xx[None] - c[:, 1, None, None]) ** 2).sqrt()) * 0.8
    mask_pred = mask_pred + torch.randn(K, H, W, generator=g) * 0.3
    n_thing = n_cls // 2
    thing_classes = [f"t{i}" for i in range(n_thing)]
    stuff_classes = (["things"] if stuff_first else []) + [f"s{i}" for i in range(n_cls - n_thing)]
    meta = types.SimpleNamespace(thing_dataset_id_to_contiguous_id={100 + i: i for i in range(n_thing)},
                                 thing_classes=thing_classes, stuff_classes=stuff_classes)
    meta.get = lambda key, default=None: getattr(meta, key, default)
    cfg = dict(prob=0.5, pano_temp=0.06, transform_eval=True, object_mask_threshold=0.3, overlap_threshold=0.6)
    images = types.SimpleNamespace(image_sizes=[image_size])
    return mask_cls, mask_pred, image_size, out_hw, meta, cfg, images


@pytest.mark.parametrize("seed,K,n_cls,stuff_first", CASES)
def test_equals_reference_function(seed, K, n_cls, stuff_first):
    mask_cls, mask_pred, image_size, out_hw, _, cfg, _ = panoptic_case(seed, K, n_cls, stuff_first)
    gold = np.load(os.path.join(GOLDEN, "panoptic_reference.npz"))
    want_seg, want_info = torch.from_numpy(gold[f"seg{seed}"]), json.loads(str(gold[f"info{seed}"]))
    n_thing = n_cls // 2
    seg, info = postprocess_panoptic(mask_cls, mask_pred, image_size, out_hw[0], out_hw[1], range(n_thing), n_thing, stuff_first, cfg)
    assert torch.equal(seg, want_seg)
    assert info == want_info
    assert len(info) > 0 or K < 4
