"""Generate golden vectors by running the REFERENCE's own Python on CPU (build container only).

Usage (in the build container, where /root/reference is mounted):
    python tests/golden/make_golden.py

Imports quant/new_pack.py (pure-torch helpers :8-129) and models/utils_quant.py (fake-quant,
:167-248, :418-432, :498-563) from /root/reference, runs them on seeded fp16 inputs and stores
inputs + outputs in tests/golden/*.npz.  The reference cannot travel to the GPU box, the
fixtures can.  Nothing here is imported at test time.
"""
import os
import sys
import warnings

import numpy as np
import torch

REF = os.environ.get("KIVI_REFERENCE_ROOT", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(REF, "quant"))
sys.path.insert(0, REF)
warnings.filterwarnings("ignore")

import new_pack as ref_pack            # noqa: E402  (reference quant/new_pack.py)
from models import utils_quant as ref_uq  # noqa: E402  (reference models/utils_quant.py)


def npy(t):
    return t.detach().cpu().numpy()


def gen_pack():
    out = {}
    for bits in (2, 4, 8):
        for g in (32, 64):
            torch.manual_seed(1000 + bits * 10 + g)
            v = torch.randn(2, 3, 5, 128, dtype=torch.float16) * 1.7 + 0.3
            code, scale, mn = ref_pack.quant_and_pack_vcache(v.clone(), g, bits)   # quant/new_pack.py:30-48
            deq = ref_pack.unpack_and_dequant_vcache(code, scale, mn, g, bits)     # :69-83
            k = torch.randn(1, 2, 128, 128, dtype=torch.float16) * 0.9 - 0.2
            kcode, kscale, kmn = ref_pack.quant_and_pack_kcache(k.clone(), g, bits)  # :8-27
            kdeq = ref_pack.unpack_and_dequant_kcache(kcode, kscale, kmn, g, bits)   # :51-66
            tag = f"b{bits}_g{g}"
            out[f"v_{tag}"] = npy(v)
            out[f"v_code_{tag}"] = npy(code)
            out[f"v_scale_{tag}"] = npy(scale.squeeze(-1))
            out[f"v_mn_{tag}"] = npy(mn.squeeze(-1))
            out[f"v_deq_{tag}"] = npy(deq)
            out[f"k_{tag}"] = npy(k)
            out[f"k_code_{tag}"] = npy(kcode)                 # [B,nh,T/fpi,D]
            out[f"k_scale_{tag}"] = npy(kscale.squeeze(-2))   # [B,nh,T/g,D]
            out[f"k_mn_{tag}"] = npy(kmn.squeeze(-2))
            out[f"k_deq_{tag}"] = npy(kdeq)
    np.savez_compressed(os.path.join(HERE, "pack_reference.npz"), **out)
    print("pack_reference.npz", len(out), "arrays")


def gen_pack_tensor():
    out = {}
    torch.manual_seed(7)
    for bits in (2, 4, 8):
        data = torch.randint(0, 2 ** bits, (2, 2, 32, 64), dtype=torch.int32)
        out[f"data_b{bits}"] = npy(data)
        out[f"pack_d2_b{bits}"] = npy(ref_pack.pack_tensor(data, bits, 2))       # :86-107
        out[f"pack_d3_b{bits}"] = npy(ref_pack.pack_tensor(data, bits, 3))
        out[f"unpack_d3_b{bits}"] = npy(ref_pack.unpack_tensor(ref_pack.pack_tensor(data, bits, 3), bits, 3)).astype(np.int32)
        out[f"unpack_d2_b{bits}"] = npy(ref_pack.unpack_tensor(ref_pack.pack_tensor(data, bits, 2), bits, 2)).astype(np.int32)
    np.savez_compressed(os.path.join(HERE, "pack_tensor_reference.npz"), **out)
    print("pack_tensor_reference.npz", len(out), "arrays")


def gen_fake_quant():
    """cfg 1 shape family: [1,H,256,128] K2V2 g32 (H = 2 keeps the fixture under 1 MB)."""
    out = {}
    torch.manual_seed(11)
    B, H, T, D, g = 1, 2, 256, 128, 32
    for bits in (2, 4):
        k = torch.randn(B, H, T, D, dtype=torch.float16)
        v = torch.randn(B, H, T, D, dtype=torch.float16)
        # per-channel K in g-token groups: models/utils_quant.py:498-521 + :533-563 (simulate=True)
        q, sc, mn = ref_uq.quantize_by_channel_and_pack_cache(k.clone(), g, bits, simulate=True)
        kdq = ref_uq.dequantize_by_channel_and_unpack_cache(q, g, k.shape, bits, sc, mn, simulate=True)
        # per-token V in g-channel groups: models/utils_quant.py:167-217
        v3 = v.transpose(1, 2).reshape(B, T, H * D)
        vdq = ref_uq.AsymGroupedQuantizer.apply(v3.clone(), None, bits, g)
        out[f"k_b{bits}"] = npy(k)
        out[f"v_b{bits}"] = npy(v)
        out[f"k_codes_b{bits}"] = npy(q)
        out[f"k_scale_b{bits}"] = npy(sc)
        out[f"k_mn_b{bits}"] = npy(mn)
        out[f"k_fake_b{bits}"] = npy(kdq)
        out[f"v_fake_b{bits}"] = npy(vdq.view(B, T, H, D).transpose(1, 2))
    np.savez_compressed(os.path.join(HERE, "fake_quant_reference.npz"), **out)
    print("fake_quant_reference.npz", len(out), "arrays")


if __name__ == "__main__":
    gen_pack()
    gen_pack_tensor()
    gen_fake_quant()
