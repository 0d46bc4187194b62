"""Generates tests/golden/ref_kernel_msda.npz: outputs of the REFERENCE's own ms_deform_attn CUDA forward kernel
(oracle/_ref/libref_msda.so, compiled for sm_100a from ape/layers/csrc/MsDeformAttn by oracle/Makefile when the reference
checkout is present) on the seeded inputs of tests/test_msda_gpu.py, at a seeded sample of queries (the full outputs are
1.8 MB and 89 MB).

Needs a GPU and a built oracle/_ref:  python tests/golden/gen_msda_ref_kernel_golden.py [output.npz]"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import msda as O  # noqa: E402
from test_msda_gpu import ref_kernel_cases  # noqa: E402


def main(path):
    assert O.have_ref_cuda(), "oracle/_ref/libref_msda.so is not built"
    arrays = {}
    for name, ins, idx in ref_kernel_cases():
        out = O.ref_cuda(*ins)
        torch.cuda.synchronize()
        arrays[name] = out[:, idx.to(out.device)].cpu().numpy()  # fp16 cases stay fp16: the kernel's own rounding
        print(name, tuple(out.shape), arrays[name].dtype, float(np.abs(arrays[name].astype(np.float32)).mean()))
    np.savez_compressed(path, **arrays)


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, "ref_kernel_msda.npz"))
