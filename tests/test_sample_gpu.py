"""Sampled decoding (kivi_sample_exchange_f32) on the GPU: parity with the float64 oracle (oracle/sample_ref.py) over the
parameter grid, greedy rows against the greedy kernel, the drawn distribution, determinism across calls / graph replays /
eager steps, generate(do_sample=True) on the tiny model, and (two GPUs) the sampling exchange against NCCL."""
import itertools
import os
import socket

import numpy as np
import pytest
import torch

from oracle import sample_ref

pytestmark = pytest.mark.gpu

GRID = list(itertools.product((0.3, 1.0, 1.7), ("0", "1", "50", "V"), (0.05, 0.9, 1.0)))   # 36 (T, k, p) rows


def _params(B, dev, T, k, p, seed, counter=1, row_offset=0):
    from kivi_b200 import glue
    return glue.SamplingParams(B, dev, row_offset=row_offset).set(temperature=T, top_k=k, top_p=p, seed=seed, counter=counter)


def _rows(V, gen, kind):
    B = len(GRID)
    # peaked rows, like a language model's: on flat rows many tiny-mass tokens fall inside the oracle's 1e-5 * Z draw band
    x = torch.randn((B, V), generator=gen, device="cuda") * 8
    if kind == "ninf":                                            # a third of every row at -inf
        x[torch.rand((B, V), generator=gen, device="cuda") < 0.33] = -float("inf")
    elif kind == "ties":                                          # few distinct values: many exact ties, also at the thresholds
        x = torch.round(x)
    return x.contiguous()


@pytest.mark.parametrize("V", [777, 32000, 128256])
def test_matches_oracle_over_the_parameter_grid(V):
    from kivi_b200 import glue
    gen = torch.Generator(device="cuda").manual_seed(V)
    T = [g[0] for g in GRID]
    k = [V if g[1] == "V" else int(g[1]) for g in GRID]
    p = [g[2] for g in GRID]
    rows = single = 0
    for kind, counter in itertools.product(("plain", "ninf", "ties"), (1, 2)):
        logits = _rows(V, gen, kind)
        B = logits.shape[0]
        sp = _params(B, logits.device, T, k, p, seed=1234 + V, counter=counter, row_offset=5)
        ids = torch.full((B,), -1, dtype=torch.long, device="cuda")
        glue.sample(logits, sp, ids)
        got = ids.cpu().numpy()
        _, acc = sample_ref.acceptable_ids(logits.cpu().numpy(), T, k, p, seed=1234 + V, counter=counter, row_offset=5)
        for b in range(B):
            assert got[b] in acc[b], (kind, counter, b, GRID[b], got[b], sorted(acc[b])[:8])
        rows += B
        single += sum(len(a) == 1 for a in acc)
    assert single >= 0.99 * rows, (single, rows)


def test_degenerate_rows_give_ids_in_range():
    from kivi_b200 import glue
    V, B = 4096, 6
    x = torch.randn((B, V), device="cuda")
    x[0, 10] = float("nan")
    x[1, :] = float("nan")
    x[2, 7] = x[2, 99] = float("inf")
    x[3, :] = -float("inf")
    x[4, 3] = -float("inf")
    x[5, :] = float("inf")
    for k, p in ((0, 1.0), (50, 0.9), (1, 0.05)):
        ids = torch.full((B,), -1, dtype=torch.long, device="cuda")
        glue.sample(x, _params(B, x.device, 1.0, k, p, seed=9), ids)
        got = ids.cpu()
        assert ((got >= 0) & (got < V)).all(), got
        assert int(got[2]) in (7, 99)                             # the +inf tokens hold all the mass


def test_greedy_rows_equal_the_greedy_kernel():
    from kivi_b200 import glue
    gen = torch.Generator(device="cuda").manual_seed(0)
    for B, V in ((32, 32000), (3, 128256), (5, 777)):             # the inputs of test_greedy_sample_matches_torch_argmax
        logits = torch.randn((B, V), generator=gen, device="cuda", dtype=torch.float16).float()
        logits[0, 5] = logits[0, 700 % V] = logits[0].max() + 1
        if B > 3:
            logits[1, 17] = logits[1, 3] = float("nan")           # the first NaN wins, as in torch.argmax
        ref = torch.full((B,), -1, dtype=torch.long, device="cuda")
        glue.greedy_sample(logits, ref)
        T = torch.zeros(B)
        T[1::2] = 1.0                                             # greedy and sampled rows in one batch
        got = torch.full((B,), -1, dtype=torch.long, device="cuda")
        fb = torch.full((B,), -1, dtype=torch.long, device="cuda")
        glue.sample(logits, _params(B, logits.device, T, 50, 0.9, seed=3), got, fb)
        assert torch.equal(got[0::2], ref[0::2]) and torch.equal(fb, got)
        assert int(got[0]) == 5


def test_drawn_distribution_matches_the_filtered_one():
    from scipy.stats import chisquare
    from kivi_b200 import glue
    V, B, T, k, p = 64, 2048, 0.8, 40, 0.9
    rng = np.random.default_rng(7)
    row = rng.standard_normal(V).astype(np.float32)
    logits = torch.from_numpy(np.tile(row, (B, 1))).cuda()
    sp = _params(B, logits.device, T, k, p, seed=2024, counter=0)
    ids = torch.empty(B, dtype=torch.long, device="cuda")
    counts = torch.zeros(V, dtype=torch.long, device="cuda")
    for _ in range(60):                                           # 122 880 draws
        sp.counter.add_(1)
        glue.sample(logits, sp, ids)
        counts += torch.bincount(ids, minlength=V)
    counts = counts.cpu().numpy()
    kept = sample_ref.kept_mask(row, T, k, p)
    assert counts[~kept].sum() == 0 and kept.sum() > 3
    e = sample_ref.masses(sample_ref.scaled(row, T)) * kept
    exp = e[kept] / e[kept].sum() * counts.sum()
    assert chisquare(counts[kept], exp).pvalue > 1e-4


def test_determinism_and_graph_replays_advance_the_counter():
    from kivi_b200 import glue
    B, V = 32, 32000
    logits = torch.randn((B, V), device="cuda") * 2
    sp = _params(B, logits.device, 1.0, 0, 1.0, seed=77, counter=5)
    a = torch.empty(B, dtype=torch.long, device="cuda")
    b = torch.empty_like(a)
    glue.sample(logits, sp, a)
    glue.sample(logits, sp, b)
    assert torch.equal(a, b)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        sp.counter.add_(1)
        glue.sample(logits, sp, b)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        sp.counter.add_(1)
        glue.sample(logits, sp, b)
    sp.counter.fill_(5)
    seen = []
    for r in range(3):
        g.replay()
        torch.cuda.synchronize()
        assert int(sp.counter) == 6 + r
        eager = torch.empty_like(a)
        glue.sample(logits, sp, eager)                            # the same counter outside the graph: the same ids
        assert torch.equal(eager, b)
        seen.append(b.clone())
    assert (seen[0] != seen[1]).sum() > B // 2 and (seen[1] != seen[2]).sum() > B // 2


def _tiny(kw, seed=0):
    from kivi_b200.llama_kivi import LlamaForCausalLM_KIVI, default_config
    cfg = default_config("tiny", **kw)
    torch.manual_seed(seed)
    return LlamaForCausalLM_KIVI(cfg).half().cuda().eval(), cfg


def test_decode_step_eager_equals_graph():
    m1, cfg = _tiny({})
    m2, _ = _tiny({})
    B, n = 4, 140
    ids = torch.randint(0, cfg.vocab_size, (B, n), device="cuda")
    toks = []
    for m, use_graph in ((m1, False), (m2, True)):
        m.init_cache(B, n + 32)
        m.set_sampling(temperature=1.0, top_k=0, top_p=0.95, seed=11)
        logits = m.prefill(ids)
        tok = logits.argmax(-1, keepdim=True)
        out = []
        for _ in range(20):
            m.decode_step(tok, use_graph=use_graph)
            tok = m.next_tokens.view(B, 1).clone()
            out.append(tok)
        toks.append(torch.cat(out, 1))
    assert torch.equal(toks[0], toks[1])


@pytest.mark.parametrize("kw", [{}, dict(num_attention_heads=4, num_key_value_heads=1, hidden_size=512, k_bits=4, v_bits=4,
                                         group_size=64, residual_length=64)])
def test_generate_do_sample(kw):
    model, cfg = _tiny(kw)
    B, n, new = 3, 140, 12
    ids = torch.randint(0, cfg.vocab_size, (B, n), device="cuda")
    a = model.generate(ids, max_new_tokens=new, do_sample=True, seed=5)
    b = model.generate(ids, max_new_tokens=new, do_sample=True, seed=5)
    c = model.generate(ids, max_new_tokens=new, do_sample=True, seed=6, top_k=0, temperature=1.5)
    assert a.shape == (B, n + new) and torch.equal(a[:, :n], ids)
    assert ((a >= 0) & (a < cfg.vocab_size)).all()
    assert torch.equal(a, b)
    assert not torch.equal(a[:, n:], c[:, n:])
    torch.manual_seed(42)
    d = model.generate(ids, max_new_tokens=new, do_sample=True)
    torch.manual_seed(42)
    assert torch.equal(d, model.generate(ids, max_new_tokens=new, do_sample=True))
    with pytest.raises(ValueError):
        model.generate(ids, max_new_tokens=new, do_sample=True, temperature=0.0)
    greedy = model.generate(ids, max_new_tokens=new)
    model.set_sampling(temperature=0.0, top_k=50, top_p=0.9, seed=1)
    assert torch.equal(model.generate(ids, max_new_tokens=new, do_sample=True), greedy)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, ws, port, out_dir):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(ws), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    from kivi_b200 import dist as kdist, glue
    kdist.init()
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    B, V = 8, 4096
    ex = kdist.PeerTokenExchange(B, dev)
    sp = glue.SamplingParams(B, dev, row_offset=rank * B).set(temperature=1.0, top_k=0, top_p=0.9, seed=99, counter=0)
    nxt = torch.zeros(B, dtype=torch.long, device=dev)
    fb = torch.zeros(B, dtype=torch.long, device=dev)
    logits = torch.randn((B, V), generator=torch.Generator(device=dev).manual_seed(100), device=dev)   # the same on both ranks
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ex.step.add_(1)
        sp.counter.add_(1)
        glue.sample(logits, sp, nxt, fb, ex)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        ex.step.add_(1)
        sp.counter.add_(1)
        glue.sample(logits, sp, nxt, fb, ex)
    differ = 0
    for it in range(6):
        g.replay()
        got = ex.tokens().clone()
        ref = torch.empty_like(nxt)
        glue.sample(logits, sp, ref)                                      # the same kernel without peers
        assert torch.equal(nxt, ref) and torch.equal(fb, nxt)
        assert torch.equal(got, kdist.gather_tokens(ref)), (rank, it)
        differ += int((got[:B] != got[B:]).sum())
    assert differ > 0                                                     # identical logits, different rows of the global batch
    torch.cuda.synchronize()
    dist.barrier()
    open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.is_available() and torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_peer_sampling_exchange_two_gpus(tmp_path):
    import torch.multiprocessing as mp
    ws = 2
    mp.spawn(_worker, args=(ws, _free_port(), str(tmp_path)), nprocs=ws, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(ws))
