"""Left-padded prompts without a GPU: the mask -> (padding, positions) conversion of the fused path against
prepare_inputs_for_generation, the masks it rejects, and the argument checks of kivi_decode_attention_padded_f16."""
import ctypes

import pytest
import torch


def _mask(rows, n):
    """rows: per row, the list of zero positions."""
    m = torch.ones(len(rows), n, dtype=torch.long)
    for b, zeros in enumerate(rows):
        m[b, zeros] = 0
    return m


@pytest.mark.parametrize("pads,n", [([0, 5, 140], 150), ([3, 0], 4), ([1], 2), ([0, 0, 7, 1], 8)])
def test_left_padding_matches_prepare_inputs(pads, n):
    from kivi_b200.llama_kivi import LlamaForCausalLM_KIVI, _left_padding, default_config
    mask = _mask([list(range(p)) for p in pads], n)
    pad, pos = _left_padding(mask)
    assert pad.tolist() == pads
    model = LlamaForCausalLM_KIVI(default_config("tiny"))
    ids = torch.zeros(len(pads), n, dtype=torch.long)
    exp = model.prepare_inputs_for_generation(ids, attention_mask=mask)["position_ids"]
    assert torch.equal(pos, exp)
    # the decode steps continue where HF's positions for one more token would be
    nxt = model.prepare_inputs_for_generation(torch.zeros(len(pads), n + 1, dtype=torch.long),
                                              attention_mask=torch.cat([mask, torch.ones(len(pads), 1, dtype=torch.long)], 1))
    assert torch.equal(nxt["position_ids"][:, -1], n - pad)
    # bool masks give the same
    pad2, pos2 = _left_padding(mask.bool())
    assert torch.equal(pad2, pad) and torch.equal(pos2, pos)


def test_unpadded_masks_need_no_padding():
    from kivi_b200.llama_kivi import _left_padding
    assert _left_padding(None) is None
    assert _left_padding(torch.ones(3, 9, dtype=torch.long)) is None


@pytest.mark.parametrize("zeros,err", [
    ([[7, 8], []], NotImplementedError),              # right padding
    ([[], [2]], NotImplementedError),                 # a hole
    ([[0, 1, 4], []], NotImplementedError),           # left padding plus a hole
    ([[], list(range(9))], ValueError),               # a row without a real token
])
def test_non_prefix_masks_are_rejected(zeros, err):
    from kivi_b200.llama_kivi import _left_padding
    with pytest.raises(err, match="left padding|real token"):
        _left_padding(_mask(zeros, 9))


def test_padded_entry_argument_validation_without_gpu():
    from kivi_b200 import build, _lib
    from kivi_b200.cache import _CacheStruct, _bind
    build.build()
    _bind()
    one = 256                                                                 # a non-NULL dummy address, never dereferenced
    c = _CacheStruct(2, 4, 2, 128, 2, 2, 32, 128, 4, 4, 129, 0, one, one, one, one, one)
    f = _lib.lib().kivi_decode_attention_padded_f16
    args = lambda **kw: [ctypes.byref(c)] + [kw.get(k, one) for k in ("q", "k", "v", "seq_start", "out", "ws")] + \
        [1 << 20, None, None, 0, kw.get("max_kv_len", 512), None]            # noqa: E731
    assert f(*args(seq_start=None)) == -6                                     # NULL seq_start
    assert f(*args(q=None)) == -6
    assert f(*args(out=None)) == -6
    assert f(*args(ws=None)) == -6
    assert f(None, *args()[1:]) == -6                                         # NULL cache
    assert f(*args(max_kv_len=0)) == -2
    assert f(*args(max_kv_len=-5)) == -2
