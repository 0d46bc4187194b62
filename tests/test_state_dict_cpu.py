"""CPU: the engine's module tree exposes exactly the reference's `state_dict` (names and shapes), so
`DetectionCheckpointer.load` (ape/engine/defaults.py:193-194) fills it by name — checked against the names and shapes of the
reference model built from its own files under the import shims, recorded by tests/golden/gen_reference_golden.py."""
import os

import numpy as np
import pytest

from ape_b200 import configs
from conftest import GOLDEN

SPECS = ["MINI", "APE_TI", "APE_L_D"]


@pytest.mark.parametrize("spec_name", SPECS)
def test_state_dict_keys_and_shapes_equal_reference(spec_name):
    from ape_b200.modeling import build_model

    gold = np.load(os.path.join(GOLDEN, "state_dict_reference.npz"))
    a = {str(k): tuple(int(d) for d in str(s).split(",") if d)
         for k, s in zip(gold[f"{spec_name}.names"], gold[f"{spec_name}.shapes"])}
    eng = build_model(getattr(configs, spec_name), num_text=16)
    b = {k: tuple(v.shape) for k, v in eng.state_dict().items()}
    assert sorted(a) == sorted(b), (sorted(set(a) - set(b))[:5], sorted(set(b) - set(a))[:5])
    assert a == b
