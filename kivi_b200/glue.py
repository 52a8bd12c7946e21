"""ctypes wrappers of the decode-step glue kernels (csrc/kivi_model.cu): residual-add + RMSNorm,
RoPE + q/k/v split, SiLU*mul, greedy sampling; and of the sampling kernel (csrc/kivi_sample.cu) with its device-side
parameters (SamplingParams).  CUDA tensors only."""
from __future__ import annotations

import ctypes

import torch

from . import _lib

_B = False


class SamplingStruct(ctypes.Structure):
    """kivi_sampling_t of include/kivi_b200.h."""
    _fields_ = [("temperature", ctypes.c_void_p), ("top_k", ctypes.c_void_p), ("top_p", ctypes.c_void_p),
                ("seed", ctypes.c_void_p), ("counter", ctypes.c_void_p), ("row_offset", ctypes.c_int32)]


def _bind():
    global _B
    if _B:
        return
    vp, i32 = ctypes.c_void_p, ctypes.c_int
    _lib.bind("kivi_add_rmsnorm_f16", i32, [vp, vp, vp, vp, i32, i32, ctypes.c_float, vp])
    _lib.bind("kivi_rope_split_f16", i32, [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp])
    _lib.bind("kivi_silu_mul_f16", i32, [vp, vp, i32, i32, vp])
    _lib.bind("kivi_greedy_sample_exchange_f32", i32, [vp, i32, i32, vp, vp, vp, i32, i32, vp, vp, vp])
    _lib.bind("kivi_sample_exchange_f32", i32, [vp, i32, i32, ctypes.POINTER(SamplingStruct), vp, vp, vp, i32, i32, vp, vp, vp])
    _B = True


def add_rmsnorm(x, residual, weight, out, eps: float):
    """residual += x (x may be None); out = weight * fp16(residual * rsqrt(mean(residual^2) + eps))."""
    _bind()
    rows, hidden = residual.shape
    _lib.check(_lib.lib().kivi_add_rmsnorm_f16(x.data_ptr() if x is not None else None, residual.data_ptr(),
                                               weight.data_ptr(), out.data_ptr(), rows, hidden, eps,
                                               _lib.stream_ptr(residual.device)), "kivi_add_rmsnorm_f16")
    return out


def rope_split(qkv, cos_table, sin_table, pos, q, k, v):
    """qkv [B,(H+2Hkv)*128] -> q [B,H,128], k [B,Hkv,128] rotated at position pos[b] (int64), v [B,Hkv,128]."""
    _bind()
    B, H, Hkv = q.shape[0], q.shape[1], k.shape[1]
    _lib.check(_lib.lib().kivi_rope_split_f16(qkv.data_ptr(), cos_table.data_ptr(), sin_table.data_ptr(), pos.data_ptr(),
                                              q.data_ptr(), k.data_ptr(), v.data_ptr(), B, H, Hkv, cos_table.shape[0],
                                              _lib.stream_ptr(qkv.device)), "kivi_rope_split_f16")


def silu_mul(gate_up, out):
    _bind()
    rows, inter = out.shape
    _lib.check(_lib.lib().kivi_silu_mul_f16(gate_up.data_ptr(), out.data_ptr(), rows, inter,
                                            _lib.stream_ptr(out.device)), "kivi_silu_mul_f16")
    return out


def greedy_sample(logits, next_local, ids_feedback=None, exchange=None):
    """next_local[b] = argmax(logits[b]) (+ copy into ids_feedback); with `exchange` (kivi_b200.dist.PeerTokenExchange) the
    same kernel also stores the ids into every rank's token buffer over NVLink and waits for the other ranks' ids."""
    _bind()
    B, V = logits.shape
    assert logits.dtype == torch.float32 and logits.is_contiguous() and next_local.dtype == torch.int64
    ex = exchange
    _lib.check(_lib.lib().kivi_greedy_sample_exchange_f32(
        logits.data_ptr(), B, V, next_local.data_ptr(), ids_feedback.data_ptr() if ids_feedback is not None else None,
        ex.peer_ptrs.data_ptr() if ex is not None else None, ex.rank if ex is not None else 0, ex.world if ex is not None else 1,
        ex.step.data_ptr() if ex is not None else None, ex.err.data_ptr() if ex is not None else None,
        _lib.stream_ptr(logits.device)), "kivi_greedy_sample_exchange_f32")
    return next_local


class SamplingParams:
    """The static device buffers of sampled decoding (kivi_sampling_t): per-row temperature, top_k, top_p, and one seed and
    one counter word.  The buffers never move, so a captured CUDA graph picks up new values set with `set()`; the caller
    increments `counter` before every `sample()` (inside the graph, like the exchange's step).
    temperature 0 makes a greedy row; top_k 0 and top_p 1 switch that filter off."""

    def __init__(self, batch: int, device, row_offset: int = 0):
        dev = torch.device(device)
        self.batch, self.row_offset = batch, int(row_offset)
        self.temperature = torch.ones(batch, dtype=torch.float32, device=dev)
        self.top_k = torch.zeros(batch, dtype=torch.int32, device=dev)
        self.top_p = torch.ones(batch, dtype=torch.float32, device=dev)
        self.seed = torch.zeros(1, dtype=torch.int64, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)
        self._struct = SamplingStruct(self.temperature.data_ptr(), self.top_k.data_ptr(), self.top_p.data_ptr(),
                                      self.seed.data_ptr(), self.counter.data_ptr(), self.row_offset)

    def _rows(self, value, dtype, name):
        t = torch.as_tensor(value, dtype=dtype).reshape(-1)
        if t.numel() == 1:
            t = t.expand(self.batch)
        if t.numel() != self.batch:
            raise ValueError(f"{name}: one value or one per row ({self.batch}), got {t.numel()}")
        return t

    def set(self, temperature=1.0, top_k=0, top_p=1.0, seed: int = 0, counter: int | None = None):
        """Copy new values into the device buffers (per-row sequences or one value for every row)."""
        t = self._rows(temperature, torch.float32, "temperature")
        k = self._rows(top_k, torch.int64, "top_k")
        p = self._rows(top_p, torch.float64, "top_p")
        if not bool((t >= 0).all()):
            raise ValueError("temperature must be >= 0 (0: a greedy row)")
        if not bool((k >= 0).all()):
            raise ValueError("top_k must be >= 0 (0: off)")
        if not bool(((p > 0) & (p <= 1)).all()):
            raise ValueError("top_p must be in (0, 1] (1: off)")
        self.temperature.copy_(t)
        self.top_k.copy_(k.clamp(max=2 ** 31 - 1).to(torch.int32))
        self.top_p.copy_(p.to(torch.float32))
        seed = int(seed) & (2 ** 64 - 1)
        self.seed.fill_(seed - 2 ** 64 if seed >= 2 ** 63 else seed)      # the uint64 word, stored in int64
        if counter is not None:
            self.counter.fill_(int(counter))
        return self


def sample(logits, params: SamplingParams, next_local, ids_feedback=None, exchange=None):
    """next_local[b] = an id drawn from row b of the fp32 logits after temperature / top-k / top-p (kivi_sample_exchange_f32,
    include/kivi_b200.h; rows with temperature 0 take the argmax) (+ copy into ids_feedback); with `exchange`
    (kivi_b200.dist.PeerTokenExchange) the ids also go to every rank's token buffer, as in greedy_sample.  The draw uses
    params.counter as it is: increment it before the call."""
    _bind()
    B, V = logits.shape
    assert logits.dtype == torch.float32 and logits.is_contiguous() and next_local.dtype == torch.int64
    assert params.batch == B and params.temperature.device == logits.device
    ex = exchange
    _lib.check(_lib.lib().kivi_sample_exchange_f32(
        logits.data_ptr(), B, V, ctypes.byref(params._struct), next_local.data_ptr(),
        ids_feedback.data_ptr() if ids_feedback is not None else None,
        ex.peer_ptrs.data_ptr() if ex is not None else None, ex.rank if ex is not None else 0, ex.world if ex is not None else 1,
        ex.step.data_ptr() if ex is not None else None, ex.err.data_ptr() if ex is not None else None,
        _lib.stream_ptr(logits.device)), "kivi_sample_exchange_f32")
    return next_local
