"""Pre-allocated KIVI cache (all layers of a model) + the fused decode-attention call.

Host-side mirror of the cache policy of LlamaFlashAttention_KIVI.forward (models/llama_kivi.py:314-455):
the reference keeps a per-layer 9-tuple that it regrows with torch.cat every step; here the buffers are
allocated once (sizes from the C ABI), the lengths live in a device int32[8] shared by all layers, and
one CUDA launch per layer does attention + cache update.  `export(layer)` returns the reference's 9-tuple.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib


class _CacheStruct(ctypes.Structure):
    """kivi_cache_t of include/kivi_b200.h"""
    _fields_ = [(n, ctypes.c_int32) for n in
                ("batch", "num_heads", "num_kv_heads", "head_dim", "k_bits", "v_bits", "group_size",
                 "residual_length", "k_cap_blocks", "v_cap_blocks", "v_res_cap", "flags")] + \
               [(n, ctypes.c_void_p) for n in ("k_store", "v_store", "k_res", "v_res", "state")]


_BOUND = False


def _bind():
    global _BOUND
    if _BOUND:
        return
    P = ctypes.POINTER(_CacheStruct)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    _lib.bind("kivi_cache_sizes", i32, [i32] * 7 + [ctypes.POINTER(i64)])
    _lib.bind("kivi_cache_prefill_f16", i32, [P, vp, vp, i32, vp])
    _lib.bind("kivi_decode_workspace_bytes", i64, [P, i32])
    _lib.bind("kivi_decode_attention_f16", i32, [P, vp, vp, vp, vp, vp, vp, i64, vp, vp, i64, i32, vp])
    _lib.bind("kivi_decode_attention_padded_f16", i32, [P, vp, vp, vp, vp, vp, vp, i64, vp, vp, i64, i32, vp])
    _lib.bind("kivi_cache_advance", i32, [P, vp])
    _lib.bind("kivi_cache_export_f16", i32, [P, i32, i32, i32, i32, i32] + [vp] * 9)
    _lib.bind("kivi_cache_import_f16", i32, [P, i32, i32, i32, i32] + [vp] * 9)
    _lib.bind("kivi_cache_read_state", i32, [P, ctypes.POINTER(ctypes.c_int32), vp])
    _BOUND = True


class KiviCache:
    """KV cache of `n_layers` attention layers: packed K/V stores + fp16 windows, fixed capacity."""

    def __init__(self, n_layers: int, batch: int, num_heads: int, num_kv_heads: int, head_dim: int = 128,
                 k_bits: int = 2, v_bits: int = 2, group_size: int = 32, residual_length: int = 128,
                 max_tokens: int = 4096, device="cuda", overlap_prologue: bool = False, gqa_chunk: int = 0):
        """overlap_prologue = KIVI_CACHE_OVERLAP_PROLOGUE of include/kivi_b200.h: promise that the kernel enqueued directly
        before every decode_attention() call never writes this cache (true inside a decoder layer, where it produces
        q / k_new / v_new), so the q.K^T launch may overlap its tail.
        gqa_chunk = KIVI_CACHE_GQA_CHUNK: query heads of a KV head that share one work unit (0 = from the geometry)."""
        _bind()
        if head_dim != 128:
            raise NotImplementedError("kivi_b200 fused decode supports head_dim 128 (all models the reference ships)")
        assert residual_length % group_size == 0                     # models/llama_kivi.py:344
        self.device = torch.device(device)
        _lib.require_cuda(torch.empty(0, device=self.device))
        self.n_layers, self.batch, self.num_heads, self.num_kv_heads = n_layers, batch, num_heads, num_kv_heads
        self.head_dim, self.k_bits, self.v_bits = head_dim, k_bits, v_bits
        self.group_size, self.residual_length, self.max_tokens = group_size, residual_length, max_tokens
        sizes = (ctypes.c_int64 * 8)()
        _lib.check(_lib.lib().kivi_cache_sizes(batch, num_kv_heads, k_bits, v_bits, group_size, residual_length,
                                               max_tokens, sizes), "kivi_cache_sizes")
        self.k_cap_blocks, self.v_cap_blocks, self.v_res_cap = int(sizes[0]), int(sizes[1]), int(sizes[2])
        self._bytes = [int(s) for s in sizes[3:7]]                    # k_store, v_store, k_res, v_res
        self.state = torch.zeros(8, dtype=torch.int32, device=self.device)
        self._bufs, self._structs = [], []
        for _ in range(n_layers):
            bufs = [torch.zeros(nb, dtype=torch.uint8, device=self.device) for nb in self._bytes]
            st = _CacheStruct(batch, num_heads, num_kv_heads, head_dim, k_bits, v_bits, group_size, residual_length,
                              self.k_cap_blocks, self.v_cap_blocks, self.v_res_cap,
                              (1 if overlap_prologue else 0) | (int(gqa_chunk) << 4),
                              *[b.data_ptr() for b in bufs], self.state.data_ptr())
            self._bufs.append(bufs)
            self._structs.append(st)
        # scratch of the decode attention (logits rows, softmax statistics, partial records, arrival counters):
        # one zero-initialised buffer shared by all layers (they run one after the other on the stream)
        nws = int(_lib.lib().kivi_decode_workspace_bytes(ctypes.byref(self._structs[0]), max_tokens))
        if nws < 0:
            _lib.check(nws, "kivi_decode_workspace_bytes")
        self._ws = torch.zeros(nws, dtype=torch.uint8, device=self.device)
        # first real position of every sequence of a left-padded batch (set_seq_start); one buffer for the cache's lifetime,
        # so that a captured decode step reads the values copied into it later
        self._seq_start = torch.zeros(batch, dtype=torch.int32, device=self.device)
        self._padded = False
        # host mirror of `state` (its evolution is deterministic)
        self.tk = self.r = self.tv = self.L = self.vhead = self.kv_len = 0

    # ------------------------------------------------------------------ bookkeeping
    def nbytes(self) -> int:
        return self.n_layers * sum(self._bytes)

    @property
    def seq_start(self) -> torch.Tensor | None:
        """The device int32 [B] of set_seq_start while padding is set, else None."""
        return self._seq_start if self._padded else None

    def set_seq_start(self, t):
        """Left padding: positions 0 .. t[b] - 1 of sequence b are padding, which decode_attention masks as an additive
        finfo(fp16).min would (kivi_decode_attention_padded_f16); negative values count as 0.  t: one int per sequence
        (list or tensor), or None to switch padding off.  The values are copied into a buffer that never moves, so a
        captured decode step picks up new values without a re-capture; switching padding on or off changes which kernel
        the step launches.  prefill() and import_tuple() switch it off."""
        if t is None:
            self._padded = False
            return
        t = torch.as_tensor(t).reshape(-1)
        if t.numel() != self.batch:
            raise ValueError(f"seq_start needs one value per sequence ({self.batch}), got {t.numel()}")
        self._seq_start.copy_(t.clamp(-2 ** 31, 2 ** 31 - 1).to(torch.int32))
        self._padded = True

    def _mirror_prefill(self, n: int):
        R = self.residual_length
        nqk = (0 if n < R else n - n % R) if n % R != 0 else n       # models/llama_kivi.py:425-434
        nqv = 0 if n <= R else n - R                                 # :442-449
        self.tk, self.r, self.tv, self.L, self.vhead, self.kv_len = nqk, n - nqk, nqv, n - nqv, 0, n

    def _mirror_advance(self):
        R = self.residual_length
        self.r += 1
        if self.r == R:                                              # :343-356
            self.tk += R
            self.r = 0
        self.L += 1
        if self.L > R:                                               # :386-399
            self.tv += 1
            self.vhead = (self.vhead + 1) % self.v_res_cap
            self.L = R
        self.kv_len += 1

    # ------------------------------------------------------------------ operations
    def prefill(self, layer: int, k: torch.Tensor, v: torch.Tensor):
        """k, v [B, Hkv, n, 128] fp16 (K post-RoPE): models/llama_kivi.py:425-452 in three launches."""
        _lib.require_cuda(k, v)
        B, Hkv, n, D = k.shape
        assert (B, Hkv, D) == (self.batch, self.num_kv_heads, self.head_dim) and v.shape == k.shape
        assert k.dtype == torch.float16 and v.dtype == torch.float16
        if n > self.max_tokens:
            raise ValueError(f"prompt of {n} tokens exceeds the cache capacity {self.max_tokens}")
        k, v = k.contiguous(), v.contiguous()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().kivi_cache_prefill_f16(ctypes.byref(self._structs[layer]), k.data_ptr(), v.data_ptr(),
                                                         n, _lib.stream_ptr(self.device)), "kivi_cache_prefill_f16")
        self._mirror_prefill(n)
        self._padded = False

    def decode_attention(self, layer: int, q: torch.Tensor, k_new: torch.Tensor, v_new: torch.Tensor,
                         mask: torch.Tensor | None = None, out: torch.Tensor | None = None,
                         dbg_logits: torch.Tensor | None = None, dbg_probs: torch.Tensor | None = None,
                         ):
        """Attention of q [B,H,128] over the cache + k_new/v_new [B,Hkv,128], then the cache update for this
        layer (two launches: q.K^T + statistics, then p.V + output + update).  Call advance() once after the last
        layer of the step.  While set_seq_start is in effect the left padding is masked and `mask` must be None."""
        _lib.require_cuda(q, k_new, v_new)
        assert q.shape == (self.batch, self.num_heads, self.head_dim) and q.dtype == torch.float16
        assert k_new.shape == (self.batch, self.num_kv_heads, self.head_dim) and v_new.shape == k_new.shape
        assert q.is_contiguous() and k_new.is_contiguous() and v_new.is_contiguous()
        if self.kv_len + 1 > self.max_tokens:
            raise ValueError("KIVI cache capacity exceeded")
        if out is None:
            out = torch.empty_like(q)
        if mask is not None:
            if self._padded:
                raise ValueError("decode_attention: pass either an additive mask or set_seq_start padding, not both")
            mask = mask.reshape(self.batch, -1).to(torch.float16).contiguous()
            assert mask.shape[1] == self.kv_len + 1
        stride = 0
        for d in (dbg_logits, dbg_probs):
            if d is not None:
                assert d.dtype == torch.float16 and d.is_contiguous() and d.shape[:2] == (self.batch, self.num_heads)
                stride = d.shape[-1]
        if self._padded:
            fn, name, extra = _lib.lib().kivi_decode_attention_padded_f16, "kivi_decode_attention_padded_f16", self._seq_start
        else:
            fn, name, extra = _lib.lib().kivi_decode_attention_f16, "kivi_decode_attention_f16", mask
        with torch.cuda.device(self.device):
            _lib.check(fn(
                ctypes.byref(self._structs[layer]), q.data_ptr(), k_new.data_ptr(), v_new.data_ptr(),
                extra.data_ptr() if extra is not None else None, out.data_ptr(),
                self._ws.data_ptr(), self._ws.numel(),
                dbg_logits.data_ptr() if dbg_logits is not None else None,
                dbg_probs.data_ptr() if dbg_probs is not None else None, stride, self.max_tokens,
                _lib.stream_ptr(self.device)), name)
        return out

    def advance(self):
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().kivi_cache_advance(ctypes.byref(self._structs[0]), _lib.stream_ptr(self.device)),
                       "kivi_cache_advance")
        self._mirror_advance()

    def read_state(self):
        """The device-side `state` words (synchronises the stream); raises if a decode kernel flagged a capacity
        violation (KIVI_STATE_ERR_CAPACITY in state[6]) and checks the host mirror."""
        host = (ctypes.c_int32 * 8)()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().kivi_cache_read_state(ctypes.byref(self._structs[0]), host, _lib.stream_ptr(self.device)),
                       "kivi_cache_read_state")
        st = list(host)
        if st[6] != 0:
            raise RuntimeError(f"kivi_b200: the decode kernels refused to run (state error word {st[6]}): the device-side "
                               f"lengths {st[:6]} exceed the capacity the cache was created with")
        return st

    def import_tuple(self, layer: int, past):
        """Load `layer` from the reference's per-layer 9-tuple (models/llama_kivi.py:454-455), the inverse of
        export(): a cache that was built by the reference's own hook (or by kivi_prefill_tuple /
        kivi_decode_attention_tuple) continues on the fused path.  All layers of a model share one `state`, so every
        layer must be imported from tuples of the same lengths."""
        kc, kfull, ks, km, vc, vfull, vs, vm, seen = past
        B, Hkv, D, g = self.batch, self.num_kv_heads, self.head_dim, self.group_size
        kf, vf = 32 // self.k_bits, 32 // self.v_bits
        tk = 0 if kc is None else kc.shape[-1] * kf
        r = 0 if kfull is None else kfull.shape[-2]
        tv = 0 if vc is None else vc.shape[-2]
        L = 0 if vfull is None else vfull.shape[-2]
        if tk + r != seen or tv + L != seen:
            raise ValueError(f"inconsistent KIVI cache tuple: tk {tk} + r {r}, tv {tv} + L {L}, kv_seq_len {seen}")
        if seen > self.max_tokens:
            raise ValueError(f"cache tuple of {seen} tokens exceeds the capacity {self.max_tokens}")

        def prep(t, shape, dtype):
            if t is None:
                return None
            _lib.require_cuda(t)
            assert tuple(t.shape) == shape and t.dtype == dtype, (tuple(t.shape), shape, t.dtype)
            return t.contiguous()
        kc = prep(kc, (B, Hkv, D, tk // kf), torch.int32)
        ks, km = prep(ks, (B, Hkv, D, tk // g), torch.float16), prep(km, (B, Hkv, D, tk // g), torch.float16)
        kfull = prep(kfull, (B, Hkv, r, D), torch.float16)
        vc = prep(vc, (B, Hkv, tv, D // vf), torch.int32)
        vs, vm = prep(vs, (B, Hkv, tv, D // g), torch.float16), prep(vm, (B, Hkv, tv, D // g), torch.float16)
        vfull = prep(vfull, (B, Hkv, L, D), torch.float16)
        ptr = lambda t: None if t is None or t.numel() == 0 else t.data_ptr()   # noqa: E731
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().kivi_cache_import_f16(
                ctypes.byref(self._structs[layer]), tk, r, tv, L, ptr(kc), ptr(ks), ptr(km), ptr(kfull),
                ptr(vc), ptr(vs), ptr(vm), ptr(vfull), _lib.stream_ptr(self.device)), "kivi_cache_import_f16")
        self.tk, self.r, self.tv, self.L, self.vhead, self.kv_len = tk, r, tv, L, 0, seen
        self._padded = False

    def export(self, layer: int):
        """The reference's per-layer 9-tuple (models/llama_kivi.py:454-455):
        (Kq_code [B,Hkv,128,tk/fpi] | None, K_full [B,Hkv,r,128] | None, K_scale, K_mn,
         Vq_code [B,Hkv,tv,128/fpi] | None, V_full [B,Hkv,L,128], V_scale, V_mn, kv_seq_len)"""
        B, Hkv, D, g = self.batch, self.num_kv_heads, self.head_dim, self.group_size
        dev = self.device
        kf, vf = 32 // self.k_bits, 32 // self.v_bits
        kc = torch.empty((B, Hkv, D, self.tk // kf), dtype=torch.int32, device=dev)
        ks = torch.empty((B, Hkv, D, self.tk // g), dtype=torch.float16, device=dev)
        km = torch.empty_like(ks)
        kfull = torch.empty((B, Hkv, self.r, D), dtype=torch.float16, device=dev)
        vc = torch.empty((B, Hkv, self.tv, D // vf), dtype=torch.int32, device=dev)
        vs = torch.empty((B, Hkv, self.tv, D // g), dtype=torch.float16, device=dev)
        vm = torch.empty_like(vs)
        vfull = torch.empty((B, Hkv, self.L, D), dtype=torch.float16, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().kivi_cache_export_f16(
                ctypes.byref(self._structs[layer]), self.tk, self.r, self.tv, self.L, self.vhead,
                kc.data_ptr(), ks.data_ptr(), km.data_ptr(), kfull.data_ptr(),
                vc.data_ptr(), vs.data_ptr(), vm.data_ptr(), vfull.data_ptr(), _lib.stream_ptr(dev)),
                "kivi_cache_export_f16")
        return (kc if self.tk > 0 else None, kfull if self.r > 0 else None, ks if self.tk > 0 else None,
                km if self.tk > 0 else None, vc if self.tv > 0 else None, vfull, vs if self.tv > 0 else None,
                vm if self.tv > 0 else None, self.kv_len)
