"""Cost of left padding on the fused decode path, on one GPU (CUDA events, after warm-up, variants alternated in rounds).

    python tools/padding_bench.py [--out padding_bench.json] [--rounds 5] [--steps 21]

Three variants of the same work:
  none    no padding: kivi_decode_attention_f16, seq_start NULL
  zeros   kivi_decode_attention_padded_f16 with seq_start all zeros (the padded kernel, nothing masked)
  uniform seq_start drawn uniformly from [0, 1024) with a fixed seed (up to 8 of a row's packed K blocks take the predicated
          epilogue; at these lengths the padding never reaches the fp16 K window)
1. ms/step of decode_step at cfg 2 (Llama-2-7B, B 32, T 4096, K2V2 g32 R128) and cfg 3 (Llama-3-8B GQA, B 64, T 8192),
   random-init weights, cache filled by prefill_synthetic (which also sets the padding and positions).  The unpadded and
   the padded step are captured once each and replayed alternately; `zeros` and `uniform` replay the same padded graph
   after a device copy of the values into the cache's seq_start buffer.
2. The per-layer attention call at the same shapes, graph-timed as in tools/microbench.py (8 back-to-back calls per replay;
   a cfg-2 layer's cache is ~0.4 GB, so consecutive calls stream from HBM, not from the 126 MB L2).
The JSON records the card's name and power limit next to the numbers, and every round's value (the spread).
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = ("none", "zeros", "uniform")
CONFIGS = (("cfg2", "llama-2-7b", 32, 4096), ("cfg3", "llama-3-8b", 64, 8192))


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the number stays meaningful with the torch name alone
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def uniform_starts(B, seed=0):
    return torch.randint(0, 1024, (B,), generator=torch.Generator().manual_seed(seed)).tolist()


def summary(t):
    out = {}
    for k, v in t.items():
        s = sorted(v)
        out[k] = {"per_round": [round(x, 4) for x in v], "median": round(s[len(s) // 2], 4), "spread": round(s[-1] - s[0], 4)}
    base = out["none"]["median"]
    for k in VARIANTS[1:]:
        out[k]["vs_none_pct"] = round(100 * (out[k]["median"] - base) / base, 3)
    return out


def graph_timer(fn, reps=8):
    """One CUDA graph of `reps` back-to-back calls; returns a function giving ms per call of one replay."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()

    def run():
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        g.replay()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps
    return run


def attention_part(key, name, B, seq, rounds):
    """One layer's decode attention call (mid-window state, no K flush in the timed calls)."""
    from kivi_b200.cache import KiviCache
    from kivi_b200.llama_kivi import default_config
    cfg = default_config(name)
    H, Hkv = cfg.num_attention_heads, cfg.num_key_value_heads
    gen = torch.Generator(device="cuda").manual_seed(0)
    cache = KiviCache(1, B, H, Hkv, 128, cfg.k_bits, cfg.v_bits, cfg.group_size, cfg.residual_length,
                      max_tokens=seq + 256, overlap_prologue=True)
    nfill = seq - 1 - cfg.residual_length // 2
    kk = torch.randn((B, Hkv, nfill, 128), generator=gen, device="cuda", dtype=torch.float16)
    vv = torch.randn((B, Hkv, nfill, 128), generator=gen, device="cuda", dtype=torch.float16)
    cache.prefill(0, kk, vv)
    del kk, vv
    q = torch.randn((B, H, 128), generator=gen, device="cuda", dtype=torch.float16)
    kn = torch.randn((B, Hkv, 128), generator=gen, device="cuda", dtype=torch.float16)
    vn = torch.randn((B, Hkv, 128), generator=gen, device="cuda", dtype=torch.float16)
    out = torch.empty_like(q)
    call = lambda: cache.decode_attention(0, q, kn, vn, out=out)          # noqa: E731
    cache.set_seq_start(None)
    run_none = graph_timer(call)
    cache.set_seq_start([0] * B)
    run_pad = graph_timer(call)
    values = {"zeros": [0] * B, "uniform": uniform_starts(B)}
    t = {k: [] for k in VARIANTS}
    for r in range(rounds):
        for k in (VARIANTS if r % 2 == 0 else VARIANTS[::-1]):
            if k != "none":
                cache.set_seq_start(values[k])
            run = run_none if k == "none" else run_pad
            run()                                                         # one untimed replay after the switch
            t[k].append(sum(run() for _ in range(3)) / 3)
    row = {"config": key, "model": name, "B": B, "kv_len": cache.kv_len + 1, "state": [cache.tk, cache.r, cache.tv, cache.L],
           "ms_per_call": summary(t)}
    print(json.dumps(row), flush=True)
    del cache
    torch.cuda.empty_cache()
    return row


def step_part(key, name, B, seq, rounds, steps):
    from kivi_b200.llama_kivi import LlamaForCausalLM_KIVI, default_config
    cfg = default_config(name)
    if seq + 64 > cfg.max_position_embeddings:
        cfg.max_position_embeddings = seq + 64
    torch.manual_seed(0)
    with torch.device("cuda"):
        model = LlamaForCausalLM_KIVI(cfg).half()
    for p_ in model.parameters():
        p_.requires_grad_(False)
    model.eval()
    total = 3 * rounds * steps + 8
    model.init_cache(B, max_tokens=seq + total)
    starts = uniform_starts(B)
    model.prefill_synthetic(seq - total // 2, seq_start=starts)           # padding + positions through the public surface
    ids = torch.randint(0, cfg.vocab_size, (B, 1), device="cuda")
    model.decode_step(ids)                                                # captures the padded step
    graphs = {True: model._graph}
    model.cache.set_seq_start(None)
    model.decode_step()                                                   # captures the unpadded step
    graphs[False] = model._graph
    values = {"zeros": [0] * B, "uniform": starts}
    t = {k: [] for k in VARIANTS}
    for r in range(rounds):
        for k in (VARIANTS if r % 2 == 0 else VARIANTS[::-1]):
            model.cache.set_seq_start(None if k == "none" else values[k])
            model._graph, model._graph_padded = graphs[k != "none"], k != "none"
            model.decode_step()                                           # one untimed replay after the switch
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps - 1):
                model.decode_step()
            b.record()
            torch.cuda.synchronize()
            t[k].append(a.elapsed_time(b) / (steps - 1))
    row = {"config": key, "model": name, "B": B, "kv_len": seq, "rounds": rounds, "steps_per_round": steps - 1,
           "ms_per_step": summary(t)}
    print(json.dumps(row), flush=True)
    del model, graphs
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=21)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("padding_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"card": card(), "attention": [], "decode_step": []}
    for key, name, B, seq in CONFIGS:
        res["attention"].append(attention_part(key, name, B, seq, a.rounds))
    for key, name, B, seq in CONFIGS:
        res["decode_step"].append(step_part(key, name, B, seq, a.rounds, a.steps))
    res["card_after"] = card()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
