"""Store the outputs of the UNMODIFIED reference CUDA extension for test_bgemv_gpu.py::test_against_reference_cuda_extension.

Usage (on a CUDA device, after oracle/build_ref.py has compiled the reference's quant/csrc into oracle/_ref/kivi_gemv.so):
    python tests/golden/make_golden_ext.py [OUT]          # default OUT: tests/golden/gemv_ext_reference.npz

Runs kivi_gemv.gemv_forward_cuda_outer_dim (quant/csrc/gemv_cuda.cu:511-557) on the seeded inputs of
tests/test_bgemv_gpu.reference_ext_cases and stores, per case, its fp16 output and the sha256 of the inputs it ran on,
so that the test needs neither the reference sources nor the extension.  Nothing here is imported at test time.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import build_ref  # noqa: E402
from tests.test_bgemv_gpu import REFERENCE_EXT_GOLDEN, reference_ext_cases  # noqa: E402


def main(out_path):
    refmod = build_ref.load()
    assert refmod is not None, f"{build_ref.SO} is missing: build it with oracle/build_ref.py"
    out = {}
    for bit in (2, 4):
        for key, (B, nh, nh_kv, IC, OC, GS), inp, _, kernel_layout, digest in reference_ext_cases(bit):
            args = [torch.from_numpy(a).cuda() for a in [inp] + kernel_layout]
            y = refmod.gemv_forward_cuda_outer_dim(*args, bit, GS, nh, nh_kv)
            torch.cuda.synchronize()
            out[key + "_out"] = y.cpu().numpy()
            out[key + "_inputs_sha256"] = np.array(digest)
    np.savez_compressed(out_path, **out)
    print(out_path, len(out), "arrays on", torch.cuda.get_device_name(0))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, REFERENCE_EXT_GOLDEN))
