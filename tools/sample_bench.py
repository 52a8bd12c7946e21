"""Cost of sampled decoding on one GPU (CUDA events, after warm-up, variants alternated in rounds).

    python tools/sample_bench.py [--out sample_bench.json] [--rounds 5] [--steps 21] [--skip-steps]

1. Kernel time, graph-timed like tools/microbench.py: the sampling kernel (kivi_sample_exchange_f32; T 0.7, top-k 50,
   top-p 0.9, and top-p 0.9 alone), the greedy kernel (kivi_greedy_sample_exchange_f32) and the torch chain of transformers'
   warpers (temperature, top-k, top-p) + torch.multinomial, at (B, V) = (32, 32000), (64, 128256), (256, 32000).
2. ms/step of decode_step, greedy against sampling (T 0.7, top-k 50, top-p 0.9), random-init cfg 2 (Llama-2-7B, B 32,
   T 4096) and cfg 3 (Llama-3-8B, B 64, T 8192) at a filled cache (prefill_synthetic).  Both steps are captured once and
   their graphs replayed alternately, `--steps` steps per variant per round.
The JSON records the card's name and power limit next to the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SAMPLING = dict(temperature=0.7, top_k=50, top_p=0.9)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # the number stays meaningful with the torch name alone
        q = f"nvidia-smi unavailable: {e}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


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


def torch_chain(logits, T, k, p, out):
    """transformers' TemperatureLogitsWarper -> TopKLogitsWarper -> TopPLogitsWarper, then multinomial."""
    s = logits / T
    s = s.masked_fill(s < torch.topk(s, k)[0][..., -1, None], -float("inf"))
    sl, si = torch.sort(s, descending=False)
    rm = sl.softmax(-1).cumsum(-1) <= (1 - p)
    rm[..., -1:] = False
    s = s.masked_fill(rm.scatter(1, si, rm), -float("inf"))
    out.copy_(torch.multinomial(s.softmax(-1), 1)[:, 0])


def kernel_part(rounds):
    from kivi_b200 import glue
    res = []
    for B, V in ((32, 32000), (64, 128256), (256, 32000)):
        logits = torch.randn((B, V), generator=torch.Generator(device="cuda").manual_seed(V + B), device="cuda") * 3
        out = torch.empty(B, dtype=torch.long, device="cuda")
        sp = glue.SamplingParams(B, "cuda").set(seed=1, **SAMPLING)
        sp_p = glue.SamplingParams(B, "cuda").set(seed=1, temperature=0.7, top_k=0, top_p=0.9)

        def smp(params):
            def f():
                params.counter.add_(1)
                glue.sample(logits, params, out)
            return f
        variants = {"sample_T0.7_k50_p0.9": graph_timer(smp(sp)), "sample_T0.7_p0.9": graph_timer(smp(sp_p)),
                    "greedy": graph_timer(lambda: glue.greedy_sample(logits, out))}
        try:
            variants["torch_chain"] = graph_timer(lambda: torch_chain(logits, 0.7, 50, 0.9, out))
        except Exception as e:
            res.append({"B": B, "V": V, "torch_chain_error": str(e)[:200]})
        t = {k: [] for k in variants}
        for _ in range(rounds):
            for k, run in variants.items():
                for _ in range(3):
                    t[k].append(run())
        row = {"B": B, "V": V}
        for k, v in t.items():
            v.sort()
            row[k + "_us_median"] = round(1e3 * v[len(v) // 2], 2)
            row[k + "_us_min"] = round(1e3 * v[0], 2)
        res.append(row)
        print(json.dumps(row), flush=True)
    return res


def step_part(name, B, seq, rounds, steps):
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
    total = 2 * rounds * steps + 8
    model.init_cache(B, max_tokens=seq + total)
    model.prefill_synthetic(seq - total // 2)
    ids = torch.randint(0, cfg.vocab_size, (B, 1), device="cuda")
    model.decode_step(ids)                                   # captures the greedy step
    graphs = {"greedy": model._graph}
    model.set_sampling(seed=0, **SAMPLING)
    model.decode_step()                                      # captures the sampling step
    graphs["sample"] = model._graph
    t = {k: [] for k in graphs}
    for r in range(rounds):
        order = list(graphs) if r % 2 == 0 else list(graphs)[::-1]
        for k in order:
            model._graph = graphs[k]
            model.decode_step()                              # one untimed replay after the switch
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(steps - 1):
                model.decode_step()
            b.record()
            torch.cuda.synchronize()
            t[k].append(a.elapsed_time(b) / (steps - 1))
    med = {k: sorted(v)[len(v) // 2] for k, v in t.items()}
    row = {"model": name, "B": B, "kv_len": seq, "rounds": rounds, "steps_per_round": steps - 1,
           "greedy_ms_per_step": [round(x, 4) for x in t["greedy"]], "sample_ms_per_step": [round(x, 4) for x in t["sample"]],
           "greedy_median_ms": round(med["greedy"], 4), "sample_median_ms": round(med["sample"], 4),
           "greedy_spread_ms": round(max(t["greedy"]) - min(t["greedy"]), 4),
           "sampling_overhead_ms": round(med["sample"] - med["greedy"], 4),
           "sampling_overhead_pct": round(100 * (med["sample"] - med["greedy"]) / med["greedy"], 3)}
    print(json.dumps(row), flush=True)
    del model, graphs
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=21)
    ap.add_argument("--skip-steps", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sample_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"card": card(), "kernels": kernel_part(a.rounds)}
    if not a.skip_steps:
        res["decode_step"] = [step_part("llama-2-7b", 32, 4096, a.rounds, a.steps),
                              step_part("llama-3-8b", 64, 8192, a.rounds, a.steps)]
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
