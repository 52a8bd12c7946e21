"""Left-padded batches on the fused path: kivi_decode_attention_padded_f16 against the additive-mask call with the equivalent
mask (bit for bit) and the oracle, inside a captured graph, and the model surface (prefill / decode_step / generate with an
HF padding mask) against the reference-style tuple path."""
import numpy as np
import pytest
import torch

from oracle import ref
from tests._util import to_np
from tests.test_decode_gpu import E2E_ATOL_FRAC, E2E_RTOL, _stage_checks, _tuple_equal

pytestmark = pytest.mark.gpu

F16_MIN = float(np.finfo(np.float16).min)


def _cache(B, H, Hkv, kb, vb, g, R, max_tokens=1024, gqa_chunk=0):
    from kivi_b200.cache import KiviCache
    return KiviCache(1, B, H, Hkv, 128, kb, vb, g, R, max_tokens, gqa_chunk=gqa_chunk)


def _twins(B, H, Hkv, kb, vb, g, R, n0, seed, gqa_chunk=0):
    """Two caches prefilled with the same prompt."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    k = torch.randn((B, Hkv, n0, 128), generator=gen, device="cuda").half()
    v = torch.randn((B, Hkv, n0, 128), generator=gen, device="cuda").half()
    caches = [_cache(B, H, Hkv, kb, vb, g, R, gqa_chunk=gqa_chunk) for _ in range(2)]
    for c in caches:
        c.prefill(0, k, v)
    return caches, gen


def _step_inputs(gen, B, H, Hkv):
    q = (torch.randn((B, H, 128), generator=gen, device="cuda") * 0.7).half()
    kn = torch.randn((B, Hkv, 128), generator=gen, device="cuda").half()
    vn = torch.randn((B, Hkv, 128), generator=gen, device="cuda").half()
    return q, kn, vn


def _equivalent_mask(starts, T):
    """The additive [B, T] fp16 mask that masks what seq_start masks: positions < max(start, 0), never the new token."""
    m = torch.zeros((len(starts), T), dtype=torch.float16, device="cuda")
    for b, s in enumerate(starts):
        m[b, :min(max(s, 0), T - 1)] = F16_MIN
    return m


def _np_tuple(t):
    return tuple(None if x is None else to_np(x) for x in t[:8]) + (t[8],)


def _tuples_identical(a, b):
    assert a[8] == b[8]
    for i in range(8):
        assert (a[i] is None) == (b[i] is None), i
        if a[i] is not None:
            assert torch.equal(a[i].view(torch.int16) if a[i].dtype == torch.float16 else a[i],
                               b[i].view(torch.int16) if b[i].dtype == torch.float16 else b[i]), f"tuple[{i}]"


GEOMS = [  # H, Hkv, kb, vb, g, R: the four bit / group / window combinations of test_prefill_matches_oracle, and GQA 4 at
    (4, 2, 2, 2, 32, 128),   # 4 bits, which reaches the 12-warp G = 4 kernels
    (4, 2, 4, 4, 64, 64),
    (4, 2, 2, 4, 32, 32),
    (4, 2, 4, 2, 128, 128),
    (8, 2, 4, 4, 64, 64),
]


@pytest.mark.parametrize("n0", [640, 20])
@pytest.mark.parametrize("H,Hkv,kb,vb,g,R", GEOMS)
@pytest.mark.parametrize("gqa_chunk", [0, 1], ids=["G-auto", "G-1"])
def test_padded_equals_mask_path(H, Hkv, kb, vb, g, R, n0, gqa_chunk):
    """Twin caches, one with seq_start and one with the equivalent additive mask rebuilt every step, over R + 2 steps (a K
    flush and V window spills with padding present): outputs, probabilities and cache tuples bit-identical, logits equal
    as fp16 values (the mask path turns -0 into +0), padding probabilities exactly 0, one step against the oracle."""
    tk = (n0 - n0 % R if n0 >= R else 0) if n0 % R else n0
    T0 = n0 + 1
    starts = [0, 1, 17, 127, 128, 129, tk, tk + 5, T0 - 2, T0, T0 + 50, -3]
    B = len(starts)
    (pc, mc), gen = _twins(B, H, Hkv, kb, vb, g, R, n0, seed=n0 + 7 * H + R + kb, gqa_chunk=gqa_chunk)
    pc.set_seq_start(starts)
    with pytest.raises(ValueError, match="not both"):
        pc.decode_attention(0, *_step_inputs(gen, B, H, Hkv), mask=_equivalent_mask(starts, T0))
    dbg = [torch.zeros((B, H, 1024), dtype=torch.float16, device="cuda") for _ in range(4)]
    for step in range(R + 2):
        T = pc.kv_len + 1
        q, kn, vn = _step_inputs(gen, B, H, Hkv)
        mask = _equivalent_mask(starts, T)
        before = _np_tuple(pc.export(0)) if step == 1 else None
        out_fast = pc.decode_attention(0, q, kn, vn).clone()              # production epilogue (padded blocks only predicated)
        out_p = pc.decode_attention(0, q, kn, vn, dbg_logits=dbg[0], dbg_probs=dbg[1])
        out_m = mc.decode_attention(0, q, kn, vn, mask=mask, dbg_logits=dbg[2], dbg_probs=dbg[3])
        torch.cuda.synchronize()
        assert torch.equal(out_fast, out_p), f"step {step}: fast and instrumented padded epilogues disagree"
        assert torch.equal(out_p.view(torch.int16), out_m.view(torch.int16)), f"step {step}: out"
        assert torch.equal(dbg[1].view(torch.int16), dbg[3].view(torch.int16)), f"step {step}: probabilities"
        assert torch.equal(dbg[0].float(), dbg[2].float()), f"step {step}: logits"
        for b, s in enumerate(starts):
            assert (dbg[1][b, :, :min(max(s, 0), T - 1)] == 0).all(), (step, b)
        if before is not None:
            mask4 = np.broadcast_to(to_np(mask)[:, None, None, :], (B, H, 1, T))
            qn, kn_, vn_ = (to_np(x)[:, :, None, :] for x in (q, kn, vn))
            _stage_checks(before, qn, kn_, vn_, g, kb, vb, R, to_np(out_p)[:, :, None, :], to_np(dbg[0])[:, :, None, :],
                          to_np(dbg[1])[:, :, None, :], mask=mask4)
            exp_out, _, exp_st = ref.decode_step(before, qn, kn_, vn_, g, kb, vb, R, mask4)
            err = np.abs(to_np(out_p)[:, :, None, :].astype(np.float64) - exp_out.astype(np.float64))
            tol = E2E_RTOL * np.abs(exp_out.astype(np.float64)) + E2E_ATOL_FRAC * np.abs(exp_out.astype(np.float64)).max()
            assert (err <= tol).all(), f"end-to-end err {err.max():.3e}"
        pc.advance()
        mc.advance()
        if before is not None:
            _tuple_equal(pc.export(0), exp_st)
    _tuples_identical(pc.export(0), mc.export(0))
    assert pc.read_state()[:6] == mc.read_state()[:6]


@pytest.mark.parametrize("H,Hkv,kb,vb,g,R", [(4, 2, 2, 2, 32, 32), (8, 2, 4, 4, 64, 64)])
def test_zero_seq_start_equals_unpadded(H, Hkv, kb, vb, g, R):
    """seq_start all zeros masks nothing: bit-identical to the NULL call (production and instrumented epilogues)."""
    B, n0 = 3, 300
    (pc, uc), gen = _twins(B, H, Hkv, kb, vb, g, R, n0, seed=11)
    pc.set_seq_start(torch.zeros(B, dtype=torch.int64))
    dbg = [torch.zeros((B, H, 512), dtype=torch.float16, device="cuda") for _ in range(4)]
    for step in range(R + 2):
        q, kn, vn = _step_inputs(gen, B, H, Hkv)
        a, b = pc.decode_attention(0, q, kn, vn).clone(), uc.decode_attention(0, q, kn, vn).clone()
        assert torch.equal(a.view(torch.int16), b.view(torch.int16)), step
        a = pc.decode_attention(0, q, kn, vn, dbg_logits=dbg[0], dbg_probs=dbg[1])
        b = uc.decode_attention(0, q, kn, vn, dbg_logits=dbg[2], dbg_probs=dbg[3])
        assert torch.equal(a.view(torch.int16), b.view(torch.int16)), step
        assert torch.equal(dbg[0].view(torch.int16), dbg[2].view(torch.int16)), step
        assert torch.equal(dbg[1].view(torch.int16), dbg[3].view(torch.int16)), step
        pc.advance()
        uc.advance()
    _tuples_identical(pc.export(0), uc.export(0))


def test_seq_start_changes_between_graph_replays():
    """The padded call captured once in a CUDA graph reads seq_start on every replay: new values copied into the buffer give
    exactly what eager calls with those values give."""
    B, H, Hkv, kb, vb, g, R, n0 = 4, 8, 2, 4, 4, 64, 64, 300
    (gc, ec), gen = _twins(B, H, Hkv, kb, vb, g, R, n0, seed=5)
    q, kn, vn = _step_inputs(gen, B, H, Hkv)
    out = torch.empty_like(q)
    for c in (gc, ec):
        c.set_seq_start([0] * B)
        c.decode_attention(0, q, kn, vn, out=out)           # warm-up (both twins: it writes past the lengths only)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        gc.decode_attention(0, q, kn, vn, out=out)
    rng = np.random.default_rng(2)
    for step in range(R + 4):
        starts = rng.integers(-2, gc.kv_len + 3, size=B).tolist()
        for c in (gc, ec):
            c.set_seq_start(starts)
        for dst, src in zip((q, kn, vn), _step_inputs(gen, B, H, Hkv)):
            dst.copy_(src)
        graph.replay()
        exp = ec.decode_attention(0, q, kn, vn)
        torch.cuda.synchronize()
        assert torch.equal(out.view(torch.int16), exp.view(torch.int16)), (step, starts)
        gc.advance()
        ec.advance()
    _tuples_identical(gc.export(0), ec.export(0))


# ---------------------------------------------------------------------------------------------------- model surface
TINY = [("tiny", {}), ("tiny", dict(num_attention_heads=4, num_key_value_heads=1, hidden_size=512, k_bits=4, v_bits=4,
                                    group_size=64, residual_length=64))]
PADS, N = [0, 5, 140], 150          # a pad longer than R and g; row 2 has 10 real tokens


def _model(name, kw, seed=0):
    from kivi_b200.llama_kivi import LlamaForCausalLM_KIVI, default_config
    cfg = default_config(name, **kw)
    torch.manual_seed(seed)
    return LlamaForCausalLM_KIVI(cfg).half().cuda().eval()


def _padded_prompt(vocab, pads=PADS, n=N, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    ids = torch.randint(0, vocab, (len(pads), n), device="cuda", generator=g)
    mask = torch.ones((len(pads), n), dtype=torch.long, device="cuda")
    for b, p in enumerate(pads):
        mask[b, :p] = 0
        ids[b, :p] = 0                                      # a pad token id, as a tokenizer would put there
    return ids, mask


@pytest.mark.parametrize("name,kw", TINY)
def test_padded_prefill_and_decode_match_tuple_model(name, kw):
    """prefill(ids, mask) + decode_step on the fused cache against the reference-style tuple path (forward with the growing
    padding mask and prepare_inputs_for_generation's positions), fed the same tokens."""
    model = _model(name, kw)
    model.fused_forward = False                             # forward() = the 9-tuple path
    B, n, steps = len(PADS), N, 40
    ids, mask = _padded_prompt(model.config.vocab_size)
    inp = model.prepare_inputs_for_generation(ids, attention_mask=mask)
    logits_t, pasts = model(ids, attention_mask=mask, position_ids=inp["position_ids"])
    model.init_cache(B, n + steps + 4)
    logits_f = model.prefill(ids, mask)
    assert model.cache.seq_start.tolist() == PADS
    assert torch.allclose(logits_f, logits_t[:, -1], rtol=2e-2, atol=2e-2)
    tok_t = logits_t[:, -1].argmax(-1, keepdim=True)
    full, m = ids, mask
    agree = 0
    for s in range(steps):
        tok = tok_t
        full = torch.cat([full, tok], 1)
        m = torch.cat([m, torch.ones_like(tok)], 1)
        inp = model.prepare_inputs_for_generation(full, past_key_values=pasts, attention_mask=m)
        lt, pasts = model(inp["input_ids"], pasts, attention_mask=m, position_ids=inp["position_ids"])
        lf = model.decode_step(tok, use_graph=(s >= 2))
        d = (lf - lt[:, -1]).abs().max().item()
        scale = lt[:, -1].abs().max().item()
        assert d <= 3e-2 * scale + 3e-2, f"step {s}: logits differ by {d} (scale {scale})"
        agree += int((lf.argmax(-1) == lt[:, -1].argmax(-1)).all())
        tok_t = lt[:, -1].argmax(-1, keepdim=True)
    assert agree >= steps - 3
    tup, ref_t = model.cache.export(0), pasts[0]
    for i in (0, 2, 3, 4, 6, 7):
        if ref_t[i] is None:
            assert tup[i] is None
        else:
            assert torch.equal(tup[i], ref_t[i].view_as(tup[i])), f"tuple[{i}]"
    assert tup[8] == ref_t[8]


@pytest.mark.parametrize("sample", [False, True], ids=["greedy", "sampled"])
@pytest.mark.parametrize("name,kw", TINY)
def test_padded_generate_matches_decode_loop(name, kw, sample):
    """generate(ids, attention_mask=mask) equals prefill + decode_step id for id; graph equals eager; HF's output layout."""
    from kivi_b200 import glue
    model = _model(name, kw, seed=1)
    ids, mask = _padded_prompt(model.config.vocab_size, seed=1)
    B, n, new = ids.shape[0], ids.shape[1], 24
    skw = dict(temperature=0.8, top_k=20, top_p=0.9, seed=7)
    gkw = dict(do_sample=True, **skw) if sample else {}
    out = model.generate(ids, attention_mask=mask, max_new_tokens=new, **gkw)
    assert out.shape == (B, n + new) and torch.equal(out[:, :n], ids)
    eager = model.generate(ids, attention_mask=mask, max_new_tokens=new, use_graph=False, **gkw)
    assert torch.equal(out, eager)
    # the same steps by hand
    if sample:
        model.set_sampling(**skw)
    else:
        model.set_sampling(None)
    logits = model.prefill(ids, mask)
    if sample:
        sp = model._sampling_params()
        sp.counter.add_(1)
        tok = glue.sample(logits.contiguous(), sp, torch.empty(B, dtype=torch.long, device="cuda")).view(B, 1)
    else:
        tok = logits.argmax(-1, keepdim=True)
    toks = [tok]
    for _ in range(new - 1):
        model.decode_step(tok)
        tok = model.next_tokens.view(B, 1).clone()
        toks.append(tok)
    assert torch.equal(out[:, n:], torch.cat(toks, 1))


def test_unpadded_generate_after_padded_matches_fresh_model():
    """A padded generate leaves nothing behind: the next unpadded generate on the same model (same cache, re-captured
    step) equals that generate on a fresh model, ids and last logits."""
    name, kw = TINY[1]
    used, fresh = _model(name, kw, seed=2), _model(name, kw, seed=2)
    ids, mask = _padded_prompt(used.config.vocab_size, seed=2)
    used.generate(ids, attention_mask=mask, max_new_tokens=16)
    used.generate(ids, attention_mask=mask, max_new_tokens=16, do_sample=True, seed=3)
    cache = used.cache
    ids2 = torch.randint(0, used.config.vocab_size, ids.shape, device="cuda")
    a = used.generate(ids2, max_new_tokens=16)
    assert used.cache is cache and cache.seq_start is None
    b = fresh.generate(ids2, max_new_tokens=16)
    assert torch.equal(a, b)
    assert torch.equal(used._logits, fresh._logits)
    a = used.generate(ids2, attention_mask=torch.ones_like(ids2), max_new_tokens=16)   # an all-ones mask is no padding
    assert torch.equal(a, b)


def test_unsupported_masks_raise():
    model = _model("tiny", {})
    ids = torch.randint(0, model.config.vocab_size, (2, 9), device="cuda")
    model.init_cache(2, 32)
    right, hole, empty = (torch.ones_like(ids) for _ in range(3))
    right[0, -2:] = 0
    hole[1, 3] = 0
    empty[1] = 0
    for fn in (lambda m: model.generate(ids, attention_mask=m, max_new_tokens=2), lambda m: model.prefill(ids, m)):
        for m in (right, hole):
            with pytest.raises(NotImplementedError, match="left padding"):
                fn(m)
        with pytest.raises(ValueError, match="real token"):
            fn(empty)
