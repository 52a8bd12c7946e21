"""Parity of the CUDA dequant-GEMVs (kivi_bgemv.cu through the C ABI / Python surface) with the oracle
(reference summation order, oracle/kivi_oracle.c) and with the stored outputs of the UNMODIFIED reference CUDA
extension on the same inputs.  Tolerance: tests/_util.py."""
import hashlib
import os

import numpy as np
import pytest
import torch

from oracle import ref
from tests._util import assert_gemv_close, l1_mass_ref_layout, to_np

pytestmark = pytest.mark.gpu


def _make_cache_ref_layout(rng, B, Hkv, K, N, g, bits, scale_mag=1.0):
    """Random fp16 [B,Hkv,K,N] quantised along N (oracle pack) -> code [B,Hkv,K,N/fpi], scale/mn [B,Hkv,K,N/g]."""
    w = (rng.standard_normal((B, Hkv, K, N)) * scale_mag).astype(np.float16)
    return ref.pack_lastdim(w, g, bits)


def _run_cuda_bmm(g, fA, code, scale, mn, bits, fn="cuda"):
    from kivi_b200 import matmul
    f = matmul.cuda_bmm_fA_qB_outer if fn == "cuda" else matmul.triton_bmm_fA_qB_outer
    out = f(g, torch.from_numpy(fA).cuda(), torch.from_numpy(code).cuda(), torch.from_numpy(scale).cuda(),
            torch.from_numpy(mn).cuda(), bits)
    torch.cuda.synchronize()
    return to_np(out)


QK_CASES = [  # (B, H, Hkv, D, Tk, g, bits)
    (2, 4, 4, 128, 128, 32, 2),
    (2, 4, 4, 128, 1024, 32, 2),
    (1, 8, 8, 128, 3968, 32, 2),      # cfg 2 token count at T=4096
    (2, 8, 2, 128, 1152, 32, 2),      # GQA ratio 4
    (1, 8, 1, 128, 640, 32, 2),       # MQA ratio 8 (two chunks of 4)
    (1, 6, 2, 128, 384, 32, 2),       # ratio 3 -> G = 1
    (1, 4, 2, 128, 2176, 64, 4),      # cfg 4 style: 4-bit g64, ratio 2
    (2, 2, 2, 128, 512, 128, 4),
    (1, 2, 2, 64, 320, 32, 2),        # head_dim 64
    (1, 2, 2, 200, 256, 64, 2),       # K not a multiple of anything nice
]


@pytest.mark.parametrize("B,H,Hkv,D,Tk,g,bits", QK_CASES)
def test_qk_shape_matches_oracle(B, H, Hkv, D, Tk, g, bits):
    """q.K^T shape of cuda_bmm_fA_qB_outer (models/llama_kivi.py:324-325): K = head_dim, N = Tk."""
    rng = np.random.default_rng(Tk * 7 + H)
    code, scale, mn = _make_cache_ref_layout(rng, B, Hkv, D, Tk, g, bits)
    q = rng.standard_normal((B, H, 1, D)).astype(np.float16)
    got = _run_cuda_bmm(g, q, code, scale, mn, bits)
    exp = ref.bmm_fA_qB_outer(g, q, code, scale, mn, bits)
    assert got.shape == exp.shape == (B, H, 1, Tk)
    assert_gemv_close(got, exp, l1_mass_ref_layout(q, scale, mn, 2 ** bits - 1), f"qk {B,H,Hkv,D,Tk,g,bits}")


SV_CASES = [  # (B, H, Hkv, Tv, D, g, bits)
    (2, 4, 4, 1, 128, 32, 2),
    (2, 4, 4, 7, 128, 32, 2),
    (1, 8, 8, 333, 128, 32, 2),
    (1, 4, 4, 3967, 128, 32, 2),      # cfg 2 at T=4096
    (2, 8, 2, 1000, 128, 32, 2),      # GQA 4
    (1, 8, 1, 129, 128, 32, 2),       # MQA 8
    (1, 4, 2, 2048, 128, 64, 4),      # 4-bit g64
    (1, 2, 2, 100, 64, 32, 2),        # head_dim 64
    (1, 2, 2, 50, 256, 128, 4),       # head_dim 256
    (1, 3, 3, 77, 96, 32, 2),         # N = 96 (3 cells)
]


@pytest.mark.parametrize("B,H,Hkv,Tv,D,g,bits", SV_CASES)
def test_sv_shape_matches_oracle(B, H, Hkv, Tv, D, g, bits):
    """p.V shape (models/llama_kivi.py:382-383): K = Tv, N = head_dim, fA = a strided slice of the probs."""
    rng = np.random.default_rng(Tv * 3 + H)
    code, scale, mn = _make_cache_ref_layout(rng, B, Hkv, Tv, D, g, bits)
    L = 5
    logits = rng.standard_normal((B, H, 1, Tv + L)).astype(np.float32) * 2
    p = (np.exp(logits) / np.exp(logits).sum(-1, keepdims=True)).astype(np.float16)
    from kivi_b200 import matmul
    pt = torch.from_numpy(p).cuda()
    out = matmul.cuda_bmm_fA_qB_outer(g, pt[:, :, :, :-L], torch.from_numpy(code).cuda(), torch.from_numpy(scale).cuda(),
                                      torch.from_numpy(mn).cuda(), bits)
    torch.cuda.synchronize()
    pq = np.ascontiguousarray(p[..., :-L])
    exp = ref.bmm_fA_qB_outer(g, pq, code, scale, mn, bits)
    assert_gemv_close(to_np(out), exp, l1_mass_ref_layout(pq, scale, mn, 2 ** bits - 1), f"sv {B,H,Hkv,Tv,D,g,bits}")


@pytest.mark.parametrize("bits,g,N", [(2, 16, 48), (2, 48, 96), (4, 8, 40), (4, 24, 48), (8, 64, 128), (8, 4, 20)])
def test_generic_group_sizes(bits, g, N):
    """Every group_size % fpi == 0 the reference kernel accepts (gemv_cuda.cu:357) plus the 8-bit Triton surface."""
    rng = np.random.default_rng(bits * 1000 + g)
    B, H, Hkv, K = 2, 4, 2, 50
    code, scale, mn = _make_cache_ref_layout(rng, B, Hkv, K, N, g, bits)
    x = rng.standard_normal((B, H, 1, K)).astype(np.float16)
    got = _run_cuda_bmm(g, x, code, scale, mn, bits, fn="triton" if bits == 8 else "cuda")
    # semantic oracle (fp64 dot of the dequantised weights) -- the C oracle covers bits 2/4 only
    c = ref.unpack_codes_lastdim(code, bits).astype(np.float64)
    w = c * np.repeat(scale.astype(np.float64), g, -1) + np.repeat(mn.astype(np.float64), g, -1)
    exp = np.einsum("bhk,bhkn->bhn", x[:, :, 0].astype(np.float64), np.repeat(w, H // Hkv, 1))[:, :, None, :]
    assert_gemv_close(got, exp.astype(np.float16), l1_mass_ref_layout(x, scale, mn, 2 ** bits - 1), "generic g")
    if bits in (2, 4):
        exp2 = ref.bmm_fA_qB_outer(g, x, code, scale, mn, bits)
        assert_gemv_close(got, exp2, l1_mass_ref_layout(x, scale, mn, 2 ** bits - 1), "generic g vs C oracle")


def _reference_test_inputs(rng, B, nh, IC, OC, GS, BIT, mqa):
    """Inputs of test_bgemv_outer_correct_mha / _mqa (quant/gemv.py:93-165), kernel layout."""
    nkv = B if mqa else B * nh
    inp = rng.standard_normal((B * nh, 1, IC)).astype(np.float16)
    w = rng.standard_normal((nkv, IC, OC)).astype(np.float16)
    code, scale, mn = ref.pack_lastdim(w, GS, BIT)                    # [nkv, IC, OC/pf], [nkv, IC, OC/g]
    qweight = np.ascontiguousarray(code.transpose(0, 2, 1))           # quant/gemv.py:113-116
    scale_t = np.ascontiguousarray(scale.transpose(0, 2, 1))
    mn_t = np.ascontiguousarray(mn.transpose(0, 2, 1))
    return inp, qweight, scale_t, mn_t


@pytest.mark.parametrize("BIT", [2, 4])
@pytest.mark.parametrize("mqa", [False, True])
def test_kernel_layout_reference_test_case(BIT, mqa):
    """The reference's own pinned case: B, nh, IC, OC = 8, 32, 739, 128, g32, seeds 0 (quant/gemv.py:14,
    :93-165, :270-276) through the `kivi_gemv` module surface; IC = 739 exercises the tail masks."""
    from kivi_b200 import kivi_gemv
    rng = np.random.default_rng(0)
    B, nh, IC, OC, GS = 8, 32, 739, 128, 32
    inp, qweight, scale, mn = _reference_test_inputs(rng, B, nh, IC, OC, GS, BIT, mqa)
    nh_kv = 1 if mqa else nh                                          # (the script's stale `False` would divide by 0)
    out = kivi_gemv.gemv_forward_cuda_outer_dim(torch.from_numpy(inp).cuda(), torch.from_numpy(qweight).cuda(),
                                                torch.from_numpy(scale).cuda(), torch.from_numpy(mn).cuda(),
                                                BIT, GS, nh, nh_kv)
    torch.cuda.synchronize()
    exp = ref.bgemv_outer_kernel_layout(inp, qweight, scale, mn, BIT, GS, nh, nh_kv)
    x = np.abs(inp.astype(np.float64))[:, 0, :]                       # [BS, IC]
    wmax = (np.abs(scale.astype(np.float64)) * (2 ** BIT - 1) + np.abs(mn.astype(np.float64))).max(1)  # [nkv, IC]
    l1 = (x * np.repeat(wmax, (B * nh) // wmax.shape[0], 0)).sum(-1)[:, None, None]
    mean_rel = assert_gemv_close(to_np(out), exp, l1, f"kernel layout bit {BIT} mqa {mqa}")
    assert mean_rel < 1e-4


REFERENCE_EXT_GOLDEN = "gemv_ext_reference.npz"


def reference_ext_cases(BIT):
    """Seeded inputs of test_against_reference_cuda_extension, case by case: (case key, (B, nh, nh_kv, IC, OC, GS),
    inp, code / scale / mn in the reference layout, the same transposed to the kernel layout, sha256 of the kernel
    inputs).  tests/golden/make_golden_ext.py runs the reference extension on exactly these."""
    rng = np.random.default_rng(1)
    for i, (B, nh, nh_kv, IC, OC, GS) in enumerate([(2, 8, 8, 739, 128, 32), (2, 8, 2, 128, 1024, 32), (1, 4, 1, 333, 128, 64)]):
        nkv = B * nh_kv
        inp = rng.standard_normal((B * nh, 1, IC)).astype(np.float16)
        w = rng.standard_normal((nkv, IC, OC)).astype(np.float16)
        code, scale, mn = ref.pack_lastdim(w, GS, BIT)
        kernel_layout = [np.ascontiguousarray(a.transpose(0, 2, 1)) for a in (code, scale, mn)]
        digest = hashlib.sha256(b"".join(a.tobytes() for a in [inp] + kernel_layout)).hexdigest()
        yield f"bit{BIT}_case{i}", (B, nh, nh_kv, IC, OC, GS), inp, (code, scale, mn), kernel_layout, digest


@pytest.mark.parametrize("BIT", [2, 4])
def test_against_reference_cuda_extension(golden_dir, BIT):
    """Kernel-vs-kernel (the only place the 1e-3 rtol bar is meaningful, SURVEY section 4): our library
    and the oracle against the outputs of the UNMODIFIED reference extension compiled for sm_100a and run on a B200
    (tests/golden/gemv_ext_reference.npz, made by tests/golden/make_golden_ext.py on the same seeded inputs)."""
    from kivi_b200 import kivi_gemv, matmul
    gold = np.load(os.path.join(golden_dir, REFERENCE_EXT_GOLDEN))
    for key, (B, nh, nh_kv, IC, OC, GS), inp, (code, scale, mn), (qw_t, sc_t, mn_t), digest in reference_ext_cases(BIT):
        assert str(gold[key + "_inputs_sha256"]) == digest, f"{key}: inputs differ from those the golden outputs were made from"
        ref_out = gold[key + "_out"]
        args = [torch.from_numpy(a).cuda() for a in (inp, qw_t, sc_t, mn_t)]
        # (1) the C oracle reproduces the reference kernel BIT FOR BIT (same order, fmaf contraction)
        orc = ref.bgemv_outer_kernel_layout(inp, qw_t, sc_t, mn_t, BIT, GS, nh, nh_kv)
        np.testing.assert_array_equal(orc.view(np.uint16), ref_out.view(np.uint16))
        # (2) our kernels, both layouts, against the reference kernel
        x = np.abs(inp.astype(np.float64))[:, 0, :]
        wmax = (np.abs(sc_t.astype(np.float64)) * (2 ** BIT - 1) + np.abs(mn_t.astype(np.float64))).max(1)
        l1 = (x * np.repeat(wmax, nh // nh_kv, 0)).sum(-1)[:, None, None]
        ours_k = kivi_gemv.gemv_forward_cuda_outer_dim(*args, BIT, GS, nh, nh_kv)
        assert_gemv_close(to_np(ours_k), ref_out, l1, "kernel layout vs reference ext")
        ours_r = matmul.cuda_bmm_fA_qB_outer(GS, args[0].view(B, nh, 1, IC), torch.from_numpy(code).cuda().view(B, nh_kv, IC, -1),
                                             torch.from_numpy(scale).cuda().view(B, nh_kv, IC, -1),
                                             torch.from_numpy(mn).cuda().view(B, nh_kv, IC, -1), BIT)
        assert_gemv_close(to_np(ours_r).reshape(B * nh, 1, OC), ref_out, l1, "reference layout vs reference ext")


@pytest.mark.parametrize("g", [64, 128])
def test_inner_gemv_matches_oracle(g):
    """gemv_forward_cuda (quant/csrc/gemv_cuda.cu:201-246): 4-bit inner-dim GEMV with padded scale rows."""
    from kivi_b200 import kivi_gemv
    rng = np.random.default_rng(g)
    Bn, IC, OC = 8, 1024, 128
    x = rng.standard_normal((Bn, IC)).astype(np.float16)
    w = rng.standard_normal((OC, IC)).astype(np.float16)
    code, scale, mn = ref.pack_lastdim(w, g, 4)
    ng = IC // g
    sf_w = (-(-(-(-ng // 8)) // 2) * 2 * 8) if g == 64 else (-(-ng // 8) * 8)
    sp = np.zeros((OC, sf_w), np.float16); sp[:, :ng] = scale
    zp = np.zeros((OC, sf_w), np.float16); zp[:, :ng] = mn
    out = kivi_gemv.gemv_forward_cuda(torch.from_numpy(x).cuda(), torch.from_numpy(code).cuda(),
                                      torch.from_numpy(sp).cuda(), torch.from_numpy(zp).cuda(), 4, g)
    torch.cuda.synchronize()
    exp = ref.gemv_inner_w4(x, code, sp, zp, g)
    l1 = (np.abs(x.astype(np.float64)).sum(-1) * (np.abs(scale.astype(np.float64)) * 15 + np.abs(mn.astype(np.float64))).max())[:, None]
    assert_gemv_close(to_np(out), exp, l1, f"inner g{g}")


def test_gemv_fwd_surface():
    """gemv_fwd (quant/gemv.py:77-90) with unpadded [OC, IC/g] scale/mn, vs fp64 semantics."""
    from kivi_b200 import gemv
    rng = np.random.default_rng(3)
    Bn, IC, OC, g, bit = 4, 512, 64, 64, 4
    x = rng.standard_normal((Bn, IC)).astype(np.float16)
    w = rng.standard_normal((OC, IC)).astype(np.float16)
    code, scale, mn = ref.pack_lastdim(w, g, bit)
    out = gemv.gemv_fwd(bit, g, torch.from_numpy(x).cuda(), torch.from_numpy(code).cuda(), torch.from_numpy(mn).cuda(),
                        torch.from_numpy(scale).cuda())
    wq = ref.unpack_codes_lastdim(code, bit).astype(np.float64) * np.repeat(scale.astype(np.float64), g, -1) + \
        np.repeat(mn.astype(np.float64), g, -1)
    exp = x.astype(np.float64) @ wq.T
    l1 = (np.abs(x.astype(np.float64)).sum(-1) * np.abs(wq).max())[:, None]
    assert_gemv_close(to_np(out), exp.astype(np.float16), l1, "gemv_fwd")
    deq = gemv.dequant_weight(torch.from_numpy(ref.unpack_codes_lastdim(code, bit)).cuda(), torch.from_numpy(scale).cuda(),
                              torch.from_numpy(mn).cuda(), g)
    np.testing.assert_array_equal(to_np(deq).view(np.uint16), ref.unpack_dequant_lastdim(code, scale, mn, g, bit).view(np.uint16))


def test_argument_errors():
    from kivi_b200 import _lib, matmul
    q = torch.zeros((1, 3, 1, 128), dtype=torch.float16, device="cuda")
    code = torch.zeros((1, 2, 128, 8), dtype=torch.int32, device="cuda")
    sc = torch.zeros((1, 2, 128, 4), dtype=torch.float16, device="cuda")
    with pytest.raises(AssertionError):                              # nh % nh_kv (quant/matmul.py:216)
        matmul.cuda_bmm_fA_qB_outer(32, q, code, sc, sc, 2)
    with pytest.raises(AssertionError):                              # bits (quant/matmul.py:215)
        matmul.cuda_bmm_fA_qB_outer(32, q[:, :2], code, sc, sc, 3)
    L = _lib.lib()
    assert L.kivi_bgemv_outer_f16(q.data_ptr(), 128, code.data_ptr(), 1024, 8, sc.data_ptr(), sc.data_ptr(), 512, 4,
                                  q.data_ptr(), 1, 2, 2, 128, 128, 2, 24, 0, None) == -4      # KIVI_ERR_GROUP
    assert L.kivi_bgemv_outer_f16(q.data_ptr(), 128, code.data_ptr(), 1024, 8, sc.data_ptr(), sc.data_ptr(), 512, 4,
                                  q.data_ptr(), 1, 2, 2, 128, 128, 2, 32, 7, None) == -7      # KIVI_ERR_LAYOUT
    assert L.kivi_bgemv_outer_f16(None, 128, code.data_ptr(), 1024, 8, sc.data_ptr(), sc.data_ptr(), 512, 4,
                                  q.data_ptr(), 1, 2, 2, 128, 128, 2, 32, 0, None) == -6      # KIVI_ERR_NULL


@pytest.mark.parametrize("kind", ["qk", "sv"])
def test_full_size_linearity(kind):
    """BASELINE cfg 2 per-layer sizes (B32 H32 T=4096: Tk=3968 / Tv=3967) -- too big for the CPU oracle, so
    parity is checked through size-independent properties: linearity in the fp16 input (x and 2x give
    exactly 2x outputs barring overflow: scaling by 2 is exact in every fp32 step) and agreement with
    the oracle on a slab of units."""
    from kivi_b200 import matmul, new_pack
    gen = torch.Generator(device="cuda").manual_seed(0)
    B, H, D, g, bits = 32, 32, 128, 32, 2
    if kind == "qk":
        T = 3968
        kT = torch.randn((B, H, D, T), generator=gen, device="cuda", dtype=torch.float16)
        code, scale, mn = new_pack.triton_quantize_and_pack_along_last_dim(kT, g, bits)
        del kT
        x = torch.randn((B, H, 1, D), generator=gen, device="cuda", dtype=torch.float16)
    else:
        T = 3967
        v = torch.randn((B, H, T, D), generator=gen, device="cuda", dtype=torch.float16)
        code, scale, mn = new_pack.triton_quantize_and_pack_along_last_dim(v, g, bits)
        del v
        x = torch.softmax(torch.randn((B, H, 1, T), generator=gen, device="cuda") * 2, -1).half()
    y1 = matmul.cuda_bmm_fA_qB_outer(g, x, code, scale, mn, bits)
    y2 = matmul.cuda_bmm_fA_qB_outer(g, x * 2, code, scale, mn, bits)
    normal = y1.abs() >= 1e-4                                         # fp16 subnormals do not scale exactly
    assert torch.equal(y2.float()[normal], y1.float()[normal] * 2)
    assert bool(((y2.float() - 2 * y1.float()).abs() <= 2.0 ** -23).all())
    sl = slice(5, 7)
    exp = ref.bmm_fA_qB_outer(g, to_np(x[sl, :4]), to_np(code[sl, :4]), to_np(scale[sl, :4]), to_np(mn[sl, :4]), bits)
    assert_gemv_close(to_np(y1[sl, :4]), exp, l1_mass_ref_layout(to_np(x[sl, :4]), to_np(scale[sl, :4]), to_np(mn[sl, :4]), 3),
                      f"full-size {kind} slab")
