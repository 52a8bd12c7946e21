"""Sampled decoding without a GPU: the oracle's Philox4x32-10 against the Random123 known-answer vectors, the oracle's kept
set against transformers' top-k / top-p warpers, and the argument checks of kivi_sample_exchange_f32."""
import ctypes

import numpy as np
import pytest

from oracle import sample_ref


@pytest.mark.parametrize("ctr,key,out", [
    ([0, 0, 0, 0], [0, 0], [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]),
    ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0],
     [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]),
])
def test_philox_known_answers(ctr, key, out):
    got = sample_ref.philox4x32_10(np.array(ctr, dtype=np.uint32), np.array(key, dtype=np.uint32))
    assert [int(v) for v in got] == out


def test_uniforms_are_in_the_open_unit_interval():
    u = sample_ref.uniforms(123, 7, np.arange(4096))
    assert (u > 0).all() and (u < 1).all() and len(np.unique(u)) > 4000
    assert not np.array_equal(u, sample_ref.uniforms(123, 8, np.arange(4096)))


def test_kept_set_matches_transformers_warpers():
    torch = pytest.importorskip("torch")
    lp = pytest.importorskip("transformers.generation.logits_process")
    rng = np.random.default_rng(0)
    for V, k, p, T in ((777, 50, 0.9, 1.0), (1000, 1000, 0.5, 0.7), (512, 7, 1.0, 1.3), (2048, 300, 0.05, 1.0),
                       (4096, 4096, 0.9, 0.3)):
        for _ in range(4):
            row = (rng.standard_normal(V) * 3).astype(np.float32)
            assert len(np.unique(row)) == V                                   # tie-free
            scores = torch.from_numpy(row)[None] / torch.tensor(T, dtype=torch.float32)
            scores = lp.TopKLogitsWarper(top_k=k)(None, scores)
            if p < 1:
                scores = lp.TopPLogitsWarper(top_p=p)(None, scores)
            hf = (scores[0] != -float("inf")).numpy()
            assert np.array_equal(sample_ref.kept_mask(row, T, k, p), hf), (V, k, p, T)


def test_argument_validation_without_gpu():
    from kivi_b200 import build, glue, _lib
    build.build()
    glue._bind()
    L = _lib.lib()
    one = 16                                                                  # a non-NULL dummy address, never dereferenced
    s = glue.SamplingStruct(one, one, one, one, one, 0)
    f = L.kivi_sample_exchange_f32
    assert f(None, 4, 32000, ctypes.byref(s), one, None, None, 0, 1, None, None, None) == -6      # NULL logits
    assert f(one, 4, 32000, None, one, None, None, 0, 1, None, None, None) == -6                 # NULL sampling struct
    assert f(one, 4, 0, ctypes.byref(s), one, None, None, 0, 1, None, None, None) == -2          # vocab <= 0
    assert f(one, 0, 32000, ctypes.byref(s), one, None, None, 0, 1, None, None, None) == -2      # batch <= 0
    assert f(one, 4, 1 << 20, ctypes.byref(s), one, None, None, 0, 1, None, None, None) == -2    # vocab too large
    s.top_p = None
    assert f(one, 4, 32000, ctypes.byref(s), one, None, None, 0, 1, None, None, None) == -6      # NULL field
