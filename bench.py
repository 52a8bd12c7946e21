#!/usr/bin/env python
"""bench.py -- decode tokens/s of Llama-2-7B with the KIVI (K2V2 g32 R128) cache on B200(s).

    python bench.py --gpus N --steps K --warmup W            # this repo (libkivi_b200 fused decode)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU fake-quant path
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's logits / ids as .npy

Metric (BASELINE.json): decode tokens/sec @ Llama-2-7B bs32 seq4k K2V2 g32 R128.  A "step" is one decode step of the
whole model for the batch: 32 x [RMSNorm, q/k/v proj, RoPE, KIVI decode attention + cache update (two libkivi_b200
launches: q.K^T, p.V), o_proj, MLP], final norm, lm_head, cache advance, greedy argmax and (N > 1) one NCCL all-gather
of the sampled ids -- all inside ONE CUDA graph.  The cache is pre-filled with synthetic K/V by the real prefill pack
kernels so that the K timed steps END at seq = 4096 tokens; weights are random-init fp16 (no checkpoints offline).
N > 1: data-parallel replicas, batch 32 per GPU (weak scaling).

One JSON line on stdout (rank 0):
  value          whole-job tokens/s, inputs resident in HBM (+ per-step CUDA-event times: median / max)
  e2e            same metric through the public API with HOST buffers (ids pinned -> H2D, logits D2H every step)
  roofline       the decode-attention call (dominant kernels of the hot path) against the measured HBM peak
  cpu_baseline   the reference's CPU fake-quant attention (oracle port of models/utils_quant.py) on the host cores
  reference_gpu  the UNMODIFIED reference CUDA extension (oracle/_ref/kivi_gemv.so, when present) at the same layer
                 shape: kernel-only and wrapper-inclusive (its transpose().contiguous() copies, quant/matmul.py:199-218)
  extra_configs  the other BASELINE.json configs, each with its own tokens/s and roofline: cfg 3 (Llama-3-8B GQA bs64
                 seq8k), cfg 4 (Mistral-7B K4V4 g64 R64 bs16 seq32k) at N = 1; cfg 5 (Llama-2-7B global batch 256 split
                 256/N per GPU) at every N.  `--no-extra` skips them.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "decode tokens/sec @ Llama-2-7B bs32 seq4k K2V2"
UNIT = "tokens/s"
MODEL_TITLES = {"llama-2-7b": "Llama-2-7B", "llama-3-8b": "Llama-3-8B (GQA)", "mistral-7b": "Mistral-7B-Instruct"}


# --------------------------------------------------------------------------------------------------
# clocks sampling (NVML polled from a thread; every sample is time-stamped and only those inside the timed region count)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20),
               ("sw_power_cap", 0x4), ("hw_power_brake_slowdown", 0x80))

    def __init__(self, gpu_index: int = 0):
        self.gpu_index, self.samples = gpu_index, []          # (t, sm_mhz, reasons mask, power W)
        self.h, self.nv, self.stop_flag, self.th, self.mx = None, None, False, None, None

    def _handle(self):
        import pynvml
        import torch
        pynvml.nvmlInit()
        self.nv = pynvml
        try:
            uuid = str(torch.cuda.get_device_properties(self.gpu_index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            return pynvml.nvmlDeviceGetHandleByUUID(uuid.encode())
        except Exception:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu_index
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu_index])
                except Exception:
                    pass
            return pynvml.nvmlDeviceGetHandleByIndex(idx)

    def _poll(self):
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                self.samples.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                     int(nv.nvmlDeviceGetCurrentClocksEventReasons(h)), nv.nvmlDeviceGetPowerUsage(h) / 1e3))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        """Started BEFORE the warm-up: the first NVML calls of a process take tens of ms."""
        try:
            self.h = self._handle()
            self.mx = float(self.nv.nvmlDeviceGetMaxClockInfo(self.h, self.nv.NVML_CLOCK_SM))
            self.th = threading.Thread(target=self._poll, daemon=True)
            self.th.start()
        except Exception:
            self.h = None

    def window(self, t0: float, t1: float):
        """Summary of the samples taken in [t0, t1] (perf_counter); widens to the 0.5 s before t1 if the region was
        shorter than a few polls."""
        if self.h is not None and self.samples:
            got = [s for s in list(self.samples) if t0 <= s[0] <= t1]
            src = "nvml 2 ms poll, samples inside the timed region"
            if len(got) < 3:
                got = [s for s in list(self.samples) if t1 - 0.5 <= s[0] <= t1 + 0.01]
                src = "nvml 2 ms poll, samples of the last 0.5 s under load (timed region shorter than 3 polls)"
            if got:
                mask = 0
                for s in got:
                    mask |= s[2]
                return {"sm_mhz": statistics.median(s[1] for s in got), "sm_min_mhz": min(s[1] for s in got),
                        "sm_max_mhz": self.mx, "reasons": sorted(n for n, bit in self.REASONS if mask & bit),
                        "power_w_max": max(s[3] for s in got), "samples": len(got), "source": src}
        try:    # fallback: one nvidia-smi query right after the timed region
            out = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,clocks.max.sm", "--format=csv,noheader,nounits",
                                  "-i", str(self.gpu_index)], capture_output=True, text=True, timeout=10).stdout.split(",")
            return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "reasons": [], "samples": 1,
                    "source": "nvidia-smi after the timed region (NVML unavailable)"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["clock sampling unavailable"], "samples": 0}

    def stop(self):
        self.stop_flag = True
        if self.th is not None:
            self.th.join(timeout=1)


# --------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's CPU fake-quant attention on host cores
# --------------------------------------------------------------------------------------------------
def cpu_fake_quant_sample(batch: int, heads: int, kv_heads: int, T: int, g: int, bits: int, reps: int):
    """One attention layer of fake-quant decode (oracle/fake_quant.py: models/utils_quant.py:167-217, :418-432,
    :498-563 restated) for `batch` sequences at kv length T: (median seconds per layer-call, cores, torch threads)."""
    import torch
    from oracle import fake_quant
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    gen = torch.Generator().manual_seed(0)
    Tq = T - T % g
    q = torch.randn((batch, heads, 1, 128), generator=gen, dtype=torch.float32)
    k = torch.randn((batch, kv_heads, Tq, 128), generator=gen, dtype=torch.float32)
    v = torch.randn((batch, kv_heads, Tq, 128), generator=gen, dtype=torch.float32)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fake_quant.fake_quant_decode_attention(q, k, v, g, bits, bits)
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), cores, torch.get_num_threads()


CPU_SAMPLE_SEQS, CPU_LAYERS = 2, 32


def cpu_sample_text(seq, t_layer, threads):
    return (f"oracle port of the reference's CPU fake-quant decode attention (models/utils_quant.py simulate paths): ONE "
            f"attention layer for {CPU_SAMPLE_SEQS} sequences x 32 heads at kv length {seq}, fp32, {threads} torch threads "
            f"({t_layer:.2f} s per layer-call); a decode step of the workload is 32 such layers, so tokens/s = "
            f"{CPU_SAMPLE_SEQS} / (t_layer x {CPU_LAYERS}); the linears are excluded (attention hot path only)")


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on this box's host cores.  A timed step =
    one bounded sample (one layer-call for 2 sequences); `ms_per_step` is its measured wall time and `units_per_step` the
    tokens that sample is worth (2 sequences x 1/32 of their layers), so value = units_per_step / seconds per step."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return 0
    cfg = workload_config(args, args.batch, args.gpus)
    t_start = time.perf_counter()
    for _ in range(max(1, min(args.warmup, 2))):
        cpu_fake_quant_sample(CPU_SAMPLE_SEQS, 32, 32, args.seq, 32, 2, 1)
    ts = []
    cores = threads = 0
    for _ in range(args.steps):
        t, cores, threads = cpu_fake_quant_sample(CPU_SAMPLE_SEQS, 32, 32, args.seq, 32, 2, 1)
        ts.append(t)
        if time.perf_counter() - t_start > 150 and len(ts) >= 3:      # bounded: the whole arm ends within a few minutes
            break
    t_layer = statistics.median(ts)
    units = CPU_SAMPLE_SEQS / CPU_LAYERS
    value = units / t_layer
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(ts),
            "warmup": args.warmup, "ms_per_step": 1e3 * t_layer, "units_per_step": units, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": cpu_sample_text(args.seq, t_layer, threads)},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "wall_s": time.perf_counter() - t_start,
            "step_ms": {"median": 1e3 * t_layer, "min": 1e3 * min(ts), "max": 1e3 * max(ts)}}
    print(json.dumps(line))
    return 0


def workload_config(args, batch, gpus, model="llama-2-7b", seq=None, kb=2, vb=2, g=32, R=128):
    seq = seq or args.seq
    return {"workload": f"{MODEL_TITLES.get(model, model)} K{kb}V{vb} g{g} residual{R}, bs{batch} per GPU, decode steps ending "
                        f"at seq {seq} (cache pre-filled by the prefill pack kernels), 1xB200 per rank",
            "batch_per_gpu": batch, "seq_len": seq, "k_bits": kb, "v_bits": vb, "group_size": g,
            "residual_length": R, "parallelism": f"dp{gpus}",
            "l2": "per-step working set (weights + KV cache, tens of GB) >> 126 MB L2: inputs larger than L2"}


# --------------------------------------------------------------------------------------------------
# one decode workload on this rank's GPU
# --------------------------------------------------------------------------------------------------
def hbm_peak():
    peak, src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peak = float(json.load(f)["hbm_gbs"])
            src = "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        pass
    return peak, src


def attention_roofline(model, cache, step_ms):
    """The decode-attention call (both kernels), back to back over all layers (cold: the layers' caches >> L2), CUDA events
    on the launching stream."""
    import torch
    cfg = model.config
    dev = cache.device
    B, H, Hkv, NL = cache.batch, cfg.num_attention_heads, cfg.num_key_value_heads, cache.n_layers
    q = torch.randn((B, H, 128), device=dev, dtype=torch.float16)
    kn = torch.randn((B, Hkv, 128), device=dev, dtype=torch.float16)
    vn = torch.randn_like(kn)
    out = torch.empty_like(q)
    while cache.r == cache.residual_length - 1:          # stay off the K-flush step (once per R steps)
        model.decode_step()
    for l in range(NL):                                  # one cold pass over all layers
        cache.decode_attention(l, q, kn, vn, out=out)
    torch.cuda.synchronize()
    reps = 3
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for l in range(NL):
            cache.decode_attention(l, q, kn, vn, out=out)
    e1.record()
    torch.cuda.synchronize()
    per_launch_ms = e0.elapsed_time(e1) / (reps * NL)
    tok_k = 128 * (cache.k_bits / 8 + 4 / cache.group_size)
    tok_v = 128 * (cache.v_bits / 8 + 4 / cache.group_size)
    U = B * Hkv
    alg_bytes = U * (cache.tk * tok_k + cache.tv * tok_v + (cache.r + cache.L) * 256) + (2 * B * H + 2 * U) * 256
    peak, peak_src = hbm_peak()
    achieved = alg_bytes / (per_launch_ms * 1e-3) / 1e9
    G = 4 if (H // Hkv) % 4 == 0 else (2 if (H // Hkv) % 2 == 0 else 1)
    cw = 12 if (cache.k_bits == 4 and G == 4) else 16                         # warps per CTA of the instantiation (kivi_attn.cuh: WarpsPerCta)
    roof = {"kernel": f"kivi_decode_attention_f16 = kivi::qk_kernel<{cache.k_bits},{G},{cache.group_size},{cw}> + "
                      f"kivi::sv_kernel<{cache.k_bits},{cache.v_bits},{G},{cache.group_size},{cw}> (q.Kq^T + window + softmax "
                      "statistics | normalise + p.Vq + window + output + cache update), timed as one call",
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "peak_source": peak_src, "launch_ms": per_launch_ms, "algorithmic_bytes_per_launch": alg_bytes,
            "state": [cache.tk, cache.r, cache.tv, cache.L], "traffic": None}
    if step_ms:
        roof["share_of_step"] = per_launch_ms * NL / step_ms
    return roof


def run_decode(model_name, B, seq, K, W, rank, ws, local, sampler=None, e2e=True, kivi=None, roofline=True, keep_outputs=False):
    """Build the model, pre-fill the cache so that the K timed steps end at kv length `seq`, time K graph-replayed steps.
    keep_outputs: res["outputs"] holds, as numpy arrays, what the last timed step returned to its caller."""
    import torch
    from kivi_b200 import dist as kdist
    from kivi_b200.llama_kivi import LlamaForCausalLM_KIVI, default_config
    dev = torch.device("cuda", local)
    cfg = default_config(model_name, **(kivi or {}))
    if seq + 64 > cfg.max_position_embeddings:
        cfg.max_position_embeddings = seq + 64
    torch.manual_seed(0)
    with torch.device(dev):
        model = LlamaForCausalLM_KIVI(cfg).half()
    for p_ in model.parameters():
        p_.requires_grad_(False)
    model.eval()
    n_e2e = K if e2e else 0
    total_steps = W + K + W + n_e2e + 8 + cfg.residual_length
    n0 = seq - (W + K)                                       # the K timed steps end at kv length `seq`
    model.init_cache(B, max_tokens=seq + total_steps + 8)
    model.prefill_synthetic(n0, seed=rank)
    cache = model.cache
    vocab = cfg.vocab_size
    Bg = B * ws
    ids = torch.randint(0, vocab, (B, 1), device=dev)
    collective = "none (1 GPU)"
    # N > 1: the ids of all replicas are exchanged inside the step's CUDA graph.  Preferred: the sampling kernel stores them
    # into the peers' symmetric buffers itself (one fused argmax + all-gather kernel over NVLink); else NCCL inside the graph;
    # else NCCL after the replay.  Whatever runs is named in the JSON line.
    attempts = [("p2p", True, "fused argmax + peer stores of the sampled ids (8 B / sequence) into every rank's symmetric buffer "
                              "(kivi_greedy_sample_exchange_f32 over NVLink, torch symmetric memory), inside the step's CUDA graph"),
                ("nccl", True, "NCCL all_gather_into_tensor of the sampled ids (8 B / sequence) inside the step's CUDA graph"),
                ("nccl", False, "NCCL all_gather_into_tensor of the sampled ids after the graph replay")] if ws > 1 else [("nccl", True, collective)]
    if os.environ.get("KIVI_BENCH_COLLECTIVE") == "nccl":
        attempts = attempts[1:]
    last_exc = None
    for mode, in_graph, text in attempts:
        try:
            ok = torch.ones(1, device=dev)
            try:
                model.enable_token_allgather(ws, in_graph=in_graph, mode=mode)
                model.decode_step(ids)                       # warm-up step 1: captures the graph
            except Exception as exc:                         # this rank failed: tell the others, all fall back together
                last_exc = exc
                ok.zero_()
            if ws > 1:
                import torch.distributed as td
                td.all_reduce(ok, op=td.ReduceOp.MIN)
            if float(ok.item()) > 0:
                collective = text
                break
            model._graph = None
            collective = None
        except Exception as exc:
            last_exc = exc
            collective = None
    if collective is None:
        raise RuntimeError(f"no token exchange worked: {last_exc}")
    for _ in range(W - 1):
        model.decode_step()                                  # feeds back its own sampled ids
    torch.cuda.synchronize()
    launches_per_step = getattr(model, "launches_per_step", None) or (2 * cfg.num_hidden_layers + 1)
    if os.environ.get("KIVI_PROFILE_STEPS"):                 # ncu --profile-from-start off: profile N steps, exit
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for _ in range(int(os.environ["KIVI_PROFILE_STEPS"])):
            model.decode_step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return None
    kdist.barrier()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    t_host0 = time.perf_counter()
    ev[0].record()
    for i in range(K):
        model.decode_step()
        ev[i + 1].record()
    torch.cuda.synchronize()
    t_host1 = time.perf_counter()
    kdist.barrier()
    ms = kdist.max_over_ranks(ev[0].elapsed_time(ev[K]))
    per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(K)]
    res = {"value": Bg * K / (ms / 1e3), "ms_per_step": ms / K,
           "step_ms": {"median": statistics.median(per_step), "min": min(per_step), "max": max(per_step),
                       "note": "per-step CUDA-event times of this rank; value uses the whole region, max over ranks"},
           "state_after_timed": [cache.tk, cache.r, cache.tv, cache.L, cache.kv_len],
           "launches_per_step": launches_per_step, "collective": collective, "global_batch": Bg,
           "clocks": sampler.window(t_host0, t_host1) if sampler is not None else None}
    all_ids = model.all_tokens
    assert all_ids.numel() == Bg
    if keep_outputs:                                         # read before the e2e steps overwrite the static buffers
        res["outputs"] = {"logits": model._logits.cpu().numpy(), "next_tokens": all_ids.cpu().numpy()}
    if ws > 1:                                               # the general path, for the record: full-logits all-gather
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        kdist.gather_logits(model._logits, Bg)
        g0.record()
        for _ in range(5):
            kdist.gather_logits(model._logits, Bg)
        g1.record()
        torch.cuda.synchronize()
        res["logits_allgather_ms"] = g0.elapsed_time(g1) / 5

    # ---- e2e: host token ids (pinned) -> H2D, step, logits D2H (pinned), every step
    if e2e:
        ids_host = torch.empty((B, 1), dtype=torch.long).pin_memory()
        logits_host = [torch.empty((B, vocab), dtype=torch.float32).pin_memory() for _ in range(2)]
        logits_stage = [torch.empty((B, vocab), dtype=torch.float32, device=dev) for _ in range(2)]
        ids_host.copy_(model.next_tokens.view(B, 1).cpu())
        ids_dev = torch.empty((B, 1), dtype=torch.long, device=dev)
        copy_stream = torch.cuda.Stream(device=dev)
        main_stream = torch.cuda.current_stream(dev)
        staged = [torch.cuda.Event() for _ in range(2)]
        copied = [torch.cuda.Event() for _ in range(2)]
        n_calls = [0]

        def step_e2e():
            # host -> device: this step's token ids (pinned); the step; device -> host: its result (the shard's logits, 4 MB,
            # through a device staging buffer on a copy stream so that the transfer overlaps the NEXT step) and the sampled
            # ids, which the host feeds back next step (the only transfer the next step has to wait for)
            i = n_calls[0] & 1
            n_calls[0] += 1
            ids_dev.copy_(ids_host, non_blocking=True)
            logits = model.decode_step(ids_dev)
            if n_calls[0] > 2:
                main_stream.wait_event(copied[i])                # the transfer of two steps ago has left this staging buffer
            logits_stage[i].copy_(logits, non_blocking=True)
            staged[i].record(main_stream)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(staged[i])
                logits_host[i].copy_(logits_stage[i], non_blocking=True)
                copied[i].record(copy_stream)
            ids_host.copy_(model.next_tokens.view(B, 1), non_blocking=True)
            main_stream.synchronize()

        for _ in range(W):
            step_e2e()
        kdist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_e2e):
            step_e2e()
        main_stream.wait_stream(copy_stream)                    # the last step's logits have landed on the host inside the timed region
        e1.record()
        torch.cuda.synchronize()
        kdist.barrier()
        ms_e2e = kdist.max_over_ranks(max(e0.elapsed_time(e1), 0.0))
        res["e2e"] = {"value": Bg * n_e2e / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": B * 8,
                      "d2h_bytes_per_step": B * vocab * 4 + B * 8, "ms_per_step": ms_e2e / n_e2e}
    if roofline and rank == 0:
        res["roofline"] = attention_roofline(model, cache, ms / K)
    res["model"] = model
    return res


def reference_gpu_timing(B, H, Hkv, T, bits, g, R):
    """The unmodified reference extension (oracle/_ref/kivi_gemv.so, built by oracle/build_ref.py) at one layer of the
    workload: gemv_forward_cuda_outer_dim kernel-only on pre-transposed operands (quant/csrc/gemv_cuda.cu:511-557) and
    wrapper-inclusive = cuda_bmm_fA_qB_outer's re-layout + kernel (quant/matmul.py:199-218, restated for timing)."""
    import torch
    try:
        from oracle import build_ref
        refmod = build_ref.load()
    except Exception as exc:
        return {"unavailable": f"{type(exc).__name__}: {exc}"}
    if refmod is None:
        return {"unavailable": "oracle/_ref/kivi_gemv.so not present (built by oracle/build_ref.py where /root/reference exists)"}
    from kivi_b200 import new_pack
    dev, D = "cuda", 128
    Tk, Tv = (T - 1) // R * R, T - 1 - R
    gen = torch.Generator(device=dev).manual_seed(0)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def timeit(fn, iters=8):
        fn()
        ts = []
        for _ in range(iters):
            flush.zero_()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        return statistics.median(ts)

    kc, ks, kz = new_pack.triton_quantize_and_pack_along_last_dim(
        torch.randn((B, Hkv, D, Tk), generator=gen, device=dev, dtype=torch.float16), g, bits)
    vc, vs, vz = new_pack.triton_quantize_and_pack_along_last_dim(
        torch.randn((B, Hkv, Tv, D), generator=gen, device=dev, dtype=torch.float16), g, bits)
    q = torch.randn((B, H, 1, D), generator=gen, device=dev, dtype=torch.float16)
    p = torch.softmax(torch.randn((B, H, 1, T), generator=gen, device=dev), -1).half()[:, :, :, :Tv]

    def wrapper(fA, qB, scales, zeros):
        Bq, nh, M, K = fA.shape
        fA2 = fA.reshape(-1, M, K).contiguous()
        qB2 = qB.reshape(-1, K, qB.shape[-1]).transpose(1, 2).contiguous()
        s2 = scales.reshape(-1, scales.shape[-2], scales.shape[-1]).transpose(1, 2).contiguous()
        z2 = zeros.reshape(-1, zeros.shape[-2], zeros.shape[-1]).transpose(1, 2).contiguous()
        return refmod.gemv_forward_cuda_outer_dim(fA2, qB2, s2, z2, bits, g, nh, qB.shape[1])

    out = {"shape": {"B": B, "H": H, "Hkv": Hkv, "T": T, "bits": bits, "g": g, "Tk": Tk, "Tv": Tv},
           "qk_wrapper_ms": timeit(lambda: wrapper(q, kc, ks, kz)), "sv_wrapper_ms": timeit(lambda: wrapper(p, vc, vs, vz))}
    q2 = q.reshape(-1, 1, D).contiguous()
    k2 = [t.reshape(-1, D, t.shape[-1]).transpose(1, 2).contiguous() for t in (kc, ks, kz)]
    out["qk_kernel_ms"] = timeit(lambda: refmod.gemv_forward_cuda_outer_dim(q2, k2[0], k2[1], k2[2], bits, g, H, Hkv))
    del k2
    p2 = p.reshape(-1, 1, Tv).contiguous()
    v2 = [t.reshape(-1, Tv, t.shape[-1]).transpose(1, 2).contiguous() for t in (vc, vs, vz)]
    out["sv_kernel_ms"] = timeit(lambda: refmod.gemv_forward_cuda_outer_dim(p2, v2[0], v2[1], v2[2], bits, g, H, Hkv))
    per_tok = D * (bits / 8 + 4 / g)
    out["qk_kernel_GBps"] = (B * Hkv * Tk * per_tok + B * H * (D + Tk) * 2) / out["qk_kernel_ms"] / 1e6
    out["sv_kernel_GBps"] = (B * Hkv * Tv * per_tok + B * H * (D + Tv) * 2) / out["sv_kernel_ms"] / 1e6
    out["two_gemv_calls_wrapper_ms"] = out["qk_wrapper_ms"] + out["sv_wrapper_ms"]
    out["note"] = ("the reference's two packed GEMV calls of one layer, single launches with an L2 flush in between (median of 8); "
                   "its decode step additionally runs the window matmuls, softmax, cats and pack launches (~30 launches / layer)")
    return out


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, outputs):
    """Write what the last timed step returned as <out_dir>/<name>.npy, so that two builds can be compared output for
    output: logits.npy (fp32 [rows, vocab], this rank's sequences), logits_rows.npy (the sequences those rows belong to)
    and next_tokens.npy (the sampled ids of every rank, as float64: exact).  When all of this rank's logits would exceed
    DUMP_LIMIT_BYTES, a fixed sample of its sequences (seed 0) is written instead."""
    import numpy as np
    logits, tokens = outputs["logits"], outputs["next_tokens"].astype(np.float64)
    rows = np.arange(logits.shape[0])
    cap = (DUMP_LIMIT_BYTES - 3 * 4096 - tokens.nbytes - logits.shape[0] * 8) // (logits.shape[1] * 4)   # 3 npy headers
    if rows.size > cap:
        rows = np.sort(np.random.default_rng(0).choice(rows.size, cap, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "logits.npy"), np.ascontiguousarray(logits[rows], np.float32))
    np.save(os.path.join(out_dir, "logits_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "next_tokens.npy"), tokens)


# --------------------------------------------------------------------------------------------------
# main arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    os.environ.setdefault("NCCL_DEBUG", "WARN")
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's version banner / logs go to stderr: stdout carries ONE JSON line
    import gc
    import torch
    from kivi_b200 import dist as kdist

    rank, ws, local = kdist.init()
    assert ws == args.gpus or ws == 1, f"--gpus {args.gpus} but WORLD_SIZE={ws}"
    torch.cuda.set_device(local)
    K, W = args.steps, max(args.warmup, 3)
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler is not None:
        sampler.start()
    B = args.batch if args.global_batch is None else args.global_batch // ws
    kivi = dict(k_bits=args.k_bits, v_bits=args.v_bits, group_size=args.group_size, residual_length=args.residual_length)
    main = run_decode(args.model, B, args.seq, K, W, rank, ws, local, sampler=sampler, kivi=kivi,
                      keep_outputs=args.dump_outputs is not None)
    if main is None:
        return 0
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, main.pop("outputs"))
    model = main.pop("model")
    mcfg = model.config
    roof = main.get("roofline")
    if roof is not None:
        try:   # DRAM bytes of the call from the committed ncu --set full capture of the same shape (NOT measured in this run)
            with open(os.path.join(ROOT, "profiles", "r02_attention_ncu.json")) as f:
                roof["traffic"] = json.load(f).get("dram_bytes_per_launch")
                roof["traffic_source"] = "profiles/r02_attention_ncu.json (ncu --set full capture of this shape; not measured in this run)"
        except Exception:
            roof["traffic_source"] = "no ncu capture committed for this build"
    shape = (B, mcfg.num_attention_heads, mcfg.num_key_value_heads)
    del model
    gc.collect()
    torch.cuda.empty_cache()

    # ---- cpu baseline (rank 0, N = 1 only): bounded sample of the same workload
    cpu = None
    if rank == 0 and ws == 1 and not args.no_cpu_baseline:
        cpu_fake_quant_sample(CPU_SAMPLE_SEQS, 32, 32, args.seq, 32, 2, 1)           # warm-up
        t_layer, cores, threads = cpu_fake_quant_sample(CPU_SAMPLE_SEQS, 32, 32, args.seq, 32, 2, 3)
        cpu = {"value": CPU_SAMPLE_SEQS / (t_layer * CPU_LAYERS), "unit": UNIT, "cores": cores, "kind": "port",
               "sample": cpu_sample_text(args.seq, t_layer, threads) + "; median of 3"}

    # ---- the reference's own GPU kernels at the same layer shape (rank 0, N = 1)
    ref_gpu = None
    if rank == 0 and ws == 1 and not args.no_reference_gpu:
        ref_gpu = reference_gpu_timing(shape[0], shape[1], shape[2], args.seq, args.k_bits, args.group_size, args.residual_length)
        if roof is not None and "two_gemv_calls_wrapper_ms" in ref_gpu:
            ref_gpu["ours_whole_attention_call_ms"] = roof["launch_ms"]
            ref_gpu["speedup_vs_two_reference_gemv_calls"] = ref_gpu["two_gemv_calls_wrapper_ms"] / roof["launch_ms"]
        gc.collect()
        torch.cuda.empty_cache()

    # ---- the other BASELINE.json configs
    extras = {}
    if not args.no_extra:
        Kx, Wx = min(K, 16), 3
        plan = []
        if ws == 1:
            plan += [("cfg3", "llama-3-8b", 64, 8192, dict(k_bits=2, v_bits=2, group_size=32, residual_length=128)),
                     ("cfg4", "mistral-7b", 16, 32768, dict(k_bits=4, v_bits=4, group_size=64, residual_length=64))]
        if 256 % ws == 0:
            plan += [("cfg5", "llama-2-7b", 256 // ws, 4096, dict(k_bits=2, v_bits=2, group_size=32, residual_length=128))]
        for key, mname, bx, sx, kv in plan:
            try:
                r = run_decode(mname, bx, sx, Kx, Wx, rank, ws, local, sampler=None, e2e=False, kivi=kv)
                r.pop("model", None)
                r.pop("clocks", None)
                r.update({"metric": f"decode tokens/sec @ {MODEL_TITLES[mname]} bs{bx * ws} seq{sx} K{kv['k_bits']}V{kv['v_bits']}",
                          "unit": UNIT, "steps": Kx, "warmup": Wx, "n_gpus": ws,
                          "scaling": "strong (global batch 256 split over the GPUs)" if key == "cfg5" else "n/a (1 GPU)",
                          "config": workload_config(args, bx, ws, mname, sx, kv["k_bits"], kv["v_bits"], kv["group_size"],
                                                    kv["residual_length"])})
                if key == "cfg4":
                    r["note"] = ("BASELINE.json writes g64 residual32; the reference rejects residual_length % group_size != 0 "
                                 "(models/mistral_kivi.py:402), so the config runs as g64 / R64 (SURVEY section 7)")
                extras[key] = r
            except Exception as exc:                         # an extra config must never take the headline line down
                extras[key] = {"error": f"{type(exc).__name__}: {exc}"}
            gc.collect()
            torch.cuda.empty_cache()
    if sampler is not None:
        sampler.stop()

    if rank == 0:
        lps = main["launches_per_step"]
        line = {"metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": ws, "steps": K, "warmup": W,
                "ms_per_step": main["ms_per_step"], "median_ms_per_step": main["step_ms"]["median"],
                "max_ms_per_step": main["step_ms"]["max"], "step_ms": main["step_ms"],
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": f"f16 (fp32 accumulate; {args.k_bits}-bit K / {args.v_bits}-bit V codes)", "data": "synthetic",
                "config": workload_config(args, B, ws, args.model, args.seq, args.k_bits, args.v_bits, args.group_size,
                                          args.residual_length),
                "clocks": main["clocks"], "e2e": main.get("e2e"),
                "e2e_note": "every step: ids pinned host -> device, the graph-replayed step, the shard's fp32 logits device -> pinned host "
                            "(through a device staging buffer on a copy stream: the 4 MB transfer overlaps the next step) and the sampled "
                            "ids device -> host, fed back from the host; the last transfer completes inside the timed region",
                "gpu_launches": lps * K,
                "gpu_launches_note": f"{lps} libkivi_b200 launches per step, counted by the library while the step was "
                                     f"captured and replayed from a CUDA graph: per layer q.K^T + p.V attention kernels, "
                                     f"add+RMSNorm x2, RoPE+split, SiLU*mul; final norm; cache advance; greedy sampling "
                                     f"(+ peer-store id exchange at N > 1).  The cuBLAS GEMMs of the same graph are not counted",
                "roofline": roof, "cpu_baseline": cpu, "reference_gpu": ref_gpu, "extra_configs": extras,
                "collective": main["collective"], "logits_allgather_ms": main.get("logits_allgather_ms"),
                "cache_state_after_timed": main["state_after_timed"],
                "note": "the timed steps end at seq 4096 and therefore include the once-per-128-steps K flush step "
                        "(tk 3968 -> 4096); the e2e steps follow at seq 4097..",
                "model": args.model, "global_batch": main["global_batch"]}
        print(json.dumps(line))
    if ws > 1:
        import torch.distributed as td
        td.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="llama-2-7b", choices=["llama-2-7b", "llama-3-8b", "mistral-7b"])
    ap.add_argument("--batch", type=int, default=32, help="sequences per GPU")
    ap.add_argument("--global-batch", type=int, default=None, help="total sequences, split evenly over the GPUs (overrides --batch)")
    ap.add_argument("--seq", type=int, default=4096)
    ap.add_argument("--k-bits", type=int, default=2, choices=[2, 4])
    ap.add_argument("--v-bits", type=int, default=2, choices=[2, 4])
    ap.add_argument("--group-size", type=int, default=32, choices=[32, 64, 128])
    ap.add_argument("--residual-length", type=int, default=128, choices=[32, 64, 128, 256])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra BASELINE configs (cfg 3 / 4 / 5)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (logits, sampled ids) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs is not None:
            ap.error("--dump-outputs applies to the default --impl ours")
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
