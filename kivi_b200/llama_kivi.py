"""Drop-in surface of the reference's models/llama_kivi.py (and, by config, models/mistral_kivi.py).

* `kivi_decode_attention_tuple`  -- the decode branch of LlamaFlashAttention_KIVI.forward
  (models/llama_kivi.py:314-399) on the reference's own 9-tuple cache, op for op, with every KIVI op
  routed to libkivi_b200 (cuda_bmm_fA_qB_outer without re-layout copies, fused pack kernel).
* `kivi_prefill_tuple`           -- the prefill split + pack (:425-455) producing that 9-tuple.
* `LlamaFlashAttention_KIVI`     -- attention module: same projections / RoPE / cache policy; the fast
  path keeps the cache in a pre-allocated `KiviCache` and runs ONE fused CUDA launch per layer per
  step (kivi_decode.cu); `past_key_value` may also be the legacy 9-tuple (then the tuple path runs).
* `LlamaForCausalLM_KIVI`        -- decoder-only LM with HF Llama parameter names (state dicts of
  LlamaForCausalLM / MistralForCausalLM load unchanged), config attrs k_bits, v_bits, group_size,
  residual_length (models/llama_kivi.py:34-38).  Host code is PyTorch (linears = cuBLAS); the decode
  step is captured in a CUDA graph.

The reference's forks star-import transformers 4.43 internals and do not import under the installed
transformers 5.5 (SURVEY 8c); this module depends on torch only and accepts any config object with the
usual Llama fields.
"""
from __future__ import annotations

import math
from types import SimpleNamespace

import torch
import torch.nn as nn
import torch.nn.functional as F

from .cache import KiviCache
from .matmul import cuda_bmm_fA_qB_outer
from .new_pack import triton_quantize_and_pack_along_last_dim


def repeat_kv(hidden_states: torch.Tensor, n_rep: int) -> torch.Tensor:
    """transformers' repeat_kv, used by the reference at models/llama_kivi.py:337,384."""
    if n_rep == 1:
        return hidden_states
    b, h, t, d = hidden_states.shape
    return hidden_states[:, :, None, :, :].expand(b, h, n_rep, t, d).reshape(b, h * n_rep, t, d)


# ---------------------------------------------------------------------------------------------------
# the reference's cache policy on its own 9-tuple (functional form of the hook)
# ---------------------------------------------------------------------------------------------------
def _cat(old, new, dim):
    return new if old is None else torch.cat([old, new], dim=dim)


def kivi_prefill_tuple(key_states, value_states, group_size, k_bits, v_bits, residual_length):
    """Prefill split + pack of models/llama_kivi.py:425-455: key/value_states [B, Hkv, n, D] -> 9-tuple.
    K: the leading n - n % R tokens are packed per channel (none if n < R), the rest stays fp16;
    V: everything but the newest R tokens is packed per token."""
    n, R = key_states.shape[-2], residual_length
    n_kq = n - n % R if n >= R else 0
    k_code = k_scale = k_mn = None
    if n_kq:
        k_code, k_scale, k_mn = triton_quantize_and_pack_along_last_dim(
            key_states[:, :, :n_kq].transpose(2, 3).contiguous(), group_size, k_bits)
    k_full = key_states[:, :, n_kq:].contiguous() if n_kq < n else None
    n_vq = max(n - R, 0)
    v_code = v_scale = v_mn = None
    if n_vq:
        v_code, v_scale, v_mn = triton_quantize_and_pack_along_last_dim(value_states[:, :, :n_vq].contiguous(),
                                                                        group_size, v_bits)
    v_full = value_states[:, :, n_vq:].contiguous() if n_vq else value_states
    return (k_code, k_full, k_scale, k_mn, v_code, v_full, v_scale, v_mn, n)


def kivi_decode_attention_tuple(query_states, key_states, value_states, past_key_value, group_size, k_bits, v_bits,
                                residual_length, attention_mask=None):
    """Decode branch of the reference hook (models/llama_kivi.py:314-399, tuple :454-455) on the
    reference's own 9-tuple, with the same rounding points; every KIVI op runs in libkivi_b200.
    query_states [B,H,1,D], key/value_states [B,Hkv,1,D] (post-RoPE) -> (attn_output [B,H,1,D], new 9-tuple)."""
    k_code, k_full, k_scale, k_mn, v_code, v_full, v_scale, v_mn, seen = past_key_value
    B, H, q_len, D = query_states.shape
    rep = H // key_states.shape[1]
    R = residual_length
    total = seen + key_states.shape[-2]

    # logits = [ q . dequant(K_packed)^T | q . K_window^T ] / sqrt(D)            (:323-341)
    k_full = _cat(k_full, key_states, 2)
    pieces = []
    if k_code is not None:
        pieces.append(cuda_bmm_fA_qB_outer(group_size, query_states, k_code, k_scale, k_mn, k_bits))
    pieces.append(torch.matmul(query_states, repeat_kv(k_full, rep).transpose(2, 3)))
    scores = (torch.cat(pieces, dim=-1) if len(pieces) > 1 else pieces[0]) / math.sqrt(D)
    if scores.shape != (B, H, q_len, total):                                     # (:358-362)
        raise ValueError(f"Attention weights should be of size {(B, H, q_len, total)}, but is {tuple(scores.shape)}")

    # a full window is packed per channel and appended along the token axis      (:343-356)
    if k_full.shape[-2] == R:
        assert R % group_size == 0
        c, sc, mn = triton_quantize_and_pack_along_last_dim(k_full.transpose(2, 3).contiguous(), group_size, k_bits)
        k_code, k_scale, k_mn, k_full = _cat(k_code, c, 3), _cat(k_scale, sc, 3), _cat(k_mn, mn, 3), None

    if attention_mask is not None:                                               # (:364-372)
        if attention_mask.shape != (B, 1, q_len, total):
            raise ValueError(f"Attention mask should be of size {(B, 1, q_len, total)}, but is {tuple(attention_mask.shape)}")
        floor = torch.tensor(torch.finfo(scores.dtype).min, device=scores.device)
        scores = torch.max(scores + attention_mask, floor)
    probs = F.softmax(scores, dim=-1, dtype=torch.float32).to(query_states.dtype)   # (:375)

    # out = probs[:tv] . dequant(V_packed) + probs[tv:] . V_window                  (:377-384)
    v_full = _cat(v_full, value_states, 2)
    L = v_full.shape[-2]
    window_part = torch.matmul(probs[..., -L:], repeat_kv(v_full, rep))
    if v_code is None:
        attn_output = window_part
    else:
        attn_output = cuda_bmm_fA_qB_outer(group_size, probs[..., :-L], v_code, v_scale, v_mn, v_bits)
        attn_output += window_part

    # the window keeps R tokens: its oldest one is packed per token                  (:386-399)
    if L > R:
        assert L == R + 1
        c, sc, mn = triton_quantize_and_pack_along_last_dim(v_full[:, :, :1].contiguous(), group_size, v_bits)
        v_code, v_scale, v_mn = _cat(v_code, c, 2), _cat(v_scale, sc, 2), _cat(v_mn, mn, 2)
        v_full = v_full[:, :, 1:].contiguous()
    return attn_output, (k_code, k_full, k_scale, k_mn, v_code, v_full, v_scale, v_mn, total)


# ---------------------------------------------------------------------------------------------------
# model
# ---------------------------------------------------------------------------------------------------
def default_config(name: str = "llama-2-7b", **kw):
    """Architecture shapes of the BASELINE configs (weights are random-init; no checkpoints offline)."""
    table = {
        "llama-2-7b": dict(hidden_size=4096, intermediate_size=11008, num_hidden_layers=32, num_attention_heads=32,
                           num_key_value_heads=32, vocab_size=32000, rope_theta=10000.0, rms_norm_eps=1e-5),
        "llama-3-8b": dict(hidden_size=4096, intermediate_size=14336, num_hidden_layers=32, num_attention_heads=32,
                           num_key_value_heads=8, vocab_size=128256, rope_theta=500000.0, rms_norm_eps=1e-5),
        "mistral-7b": dict(hidden_size=4096, intermediate_size=14336, num_hidden_layers=32, num_attention_heads=32,
                           num_key_value_heads=8, vocab_size=32000, rope_theta=1000000.0, rms_norm_eps=1e-5),
        "tiny": dict(hidden_size=256, intermediate_size=512, num_hidden_layers=2, num_attention_heads=2,
                     num_key_value_heads=2, vocab_size=512, rope_theta=10000.0, rms_norm_eps=1e-5),
    }
    cfg = dict(table[name], k_bits=2, v_bits=2, group_size=32, residual_length=128, use_flash=True,
               max_position_embeddings=32768 + 1024)
    cfg.update(kw)
    return SimpleNamespace(**cfg)


class LlamaRMSNorm(nn.Module):
    def __init__(self, hidden_size, eps):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(hidden_size))
        self.variance_epsilon = eps

    def forward(self, x):
        return F.rms_norm(x, (x.shape[-1],), self.weight, self.variance_epsilon)


def _rope_tables(head_dim, max_pos, theta, device):
    inv_freq = 1.0 / (theta ** (torch.arange(0, head_dim, 2, dtype=torch.float32, device=device) / head_dim))
    freqs = torch.outer(torch.arange(max_pos, dtype=torch.float32, device=device), inv_freq)
    emb = torch.cat((freqs, freqs), dim=-1)
    return emb.cos().half(), emb.sin().half()


def _rotate_half(x):
    x1, x2 = x[..., : x.shape[-1] // 2], x[..., x.shape[-1] // 2:]
    return torch.cat((-x2, x1), dim=-1)


class LlamaFlashAttention_KIVI(nn.Module):
    """Attention layer of the reference (models/llama_kivi.py:264-466), KIVI ops on libkivi_b200."""

    def __init__(self, config, layer_idx: int = 0):
        super().__init__()
        self.config = config
        self.layer_idx = layer_idx
        self.hidden_size = config.hidden_size
        self.num_heads = config.num_attention_heads
        self.head_dim = self.hidden_size // self.num_heads
        self.num_key_value_heads = config.num_key_value_heads
        self.num_key_value_groups = self.num_heads // self.num_key_value_heads
        self.k_bits, self.v_bits = config.k_bits, config.v_bits            # models/llama_kivi.py:34-38
        self.group_size, self.residual_length = config.group_size, config.residual_length
        bias = getattr(config, "attention_bias", False)
        self.q_proj = nn.Linear(self.hidden_size, self.num_heads * self.head_dim, bias=bias)
        self.k_proj = nn.Linear(self.hidden_size, self.num_key_value_heads * self.head_dim, bias=bias)
        self.v_proj = nn.Linear(self.hidden_size, self.num_key_value_heads * self.head_dim, bias=bias)
        self.o_proj = nn.Linear(self.num_heads * self.head_dim, self.hidden_size, bias=bias)

    def _qkv(self, hidden_states, cos, sin):
        bsz, q_len, _ = hidden_states.shape
        q = self.q_proj(hidden_states).view(bsz, q_len, self.num_heads, self.head_dim).transpose(1, 2)
        k = self.k_proj(hidden_states).view(bsz, q_len, self.num_key_value_heads, self.head_dim).transpose(1, 2)
        v = self.v_proj(hidden_states).view(bsz, q_len, self.num_key_value_heads, self.head_dim).transpose(1, 2)
        q = q * cos + _rotate_half(q) * sin                                 # apply_rotary_pos_emb (:311)
        k = k * cos + _rotate_half(k) * sin
        return q, k, v

    def _prompt_attention(self, q, k, v, attention_mask):
        """Attention over the prompt itself (the reference calls flash-attn here, models/llama_kivi.py:401-423; off the
        decode hot path): causal, plus the additive mask [B, 1, q_len, q_len] when the batch is padded."""
        kk, vv = repeat_kv(k, self.num_key_value_groups), repeat_kv(v, self.num_key_value_groups)
        if attention_mask is None:
            return F.scaled_dot_product_attention(q, kk, vv, is_causal=True)
        return F.scaled_dot_product_attention(q, kk, vv, attn_mask=attention_mask.to(q.dtype))

    def forward(self, hidden_states, cos, sin, past_key_value=None, attention_mask=None):
        """hidden_states [B, q_len, hidden]; cos/sin broadcastable to [B, 1, q_len, D].
        past_key_value: None (prefill, returns a 9-tuple), a 9-tuple (reference semantics), or a
        (KiviCache, layer) pair (fused path; prefill fills it, decode is one launch).
        attention_mask: None or additive [B, 1, q_len, kv_len] (models/llama_kivi.py:364-372)."""
        bsz, q_len, _ = hidden_states.shape
        q, k, v = self._qkv(hidden_states, cos, sin)
        fused = isinstance(past_key_value, tuple) and len(past_key_value) == 2 and isinstance(past_key_value[0], KiviCache)
        if fused:
            cache, layer = past_key_value
            if q_len > 1:                                                   # prefill (:401-452)
                attn_output = self._prompt_attention(q, k, v, attention_mask)
                cache.prefill(layer, k, v)
                attn_output = attn_output.transpose(1, 2).reshape(bsz, q_len, self.hidden_size)
            else:                                                           # decode (:314-399), one launch
                out = cache.decode_attention(layer, q.reshape(bsz, self.num_heads, self.head_dim).contiguous(),
                                             k.reshape(bsz, self.num_key_value_heads, self.head_dim).contiguous(),
                                             v.reshape(bsz, self.num_key_value_heads, self.head_dim).contiguous(),
                                             mask=attention_mask)
                attn_output = out.view(bsz, 1, self.hidden_size)
            return self.o_proj(attn_output), None, past_key_value
        if past_key_value is not None:                                      # reference 9-tuple, decode
            attn_output, past = kivi_decode_attention_tuple(q, k, v, past_key_value, self.group_size, self.k_bits,
                                                            self.v_bits, self.residual_length, attention_mask)
            attn_output = attn_output.transpose(1, 2).contiguous()
        else:                                                               # prefill -> 9-tuple
            attn_output = self._prompt_attention(q, k, v, attention_mask).transpose(1, 2)
            past = kivi_prefill_tuple(k, v, self.group_size, self.k_bits, self.v_bits, self.residual_length)
        attn_output = attn_output.reshape(bsz, q_len, self.hidden_size)
        return self.o_proj(attn_output), None, past


LlamaAttention_KIVI = LlamaFlashAttention_KIVI      # models/llama_kivi.py:19 (unreachable in the reference: ctor asserts use_flash)


class LlamaMLP(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.gate_proj = nn.Linear(config.hidden_size, config.intermediate_size, bias=False)
        self.up_proj = nn.Linear(config.hidden_size, config.intermediate_size, bias=False)
        self.down_proj = nn.Linear(config.intermediate_size, config.hidden_size, bias=False)

    def forward(self, x):
        return self.down_proj(F.silu(self.gate_proj(x)) * self.up_proj(x))


class LlamaDecoderLayer_KIVI(nn.Module):
    def __init__(self, config, layer_idx):
        super().__init__()
        self.self_attn = LlamaFlashAttention_KIVI(config, layer_idx)
        self.mlp = LlamaMLP(config)
        self.input_layernorm = LlamaRMSNorm(config.hidden_size, config.rms_norm_eps)
        self.post_attention_layernorm = LlamaRMSNorm(config.hidden_size, config.rms_norm_eps)

    def forward(self, hidden_states, cos, sin, past_key_value=None, attention_mask=None):
        residual = hidden_states
        h, _, past = self.self_attn(self.input_layernorm(hidden_states), cos, sin, past_key_value, attention_mask)
        hidden_states = residual + h
        hidden_states = hidden_states + self.mlp(self.post_attention_layernorm(hidden_states))
        return hidden_states, past


class LlamaModel_KIVI(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.embed_tokens = nn.Embedding(config.vocab_size, config.hidden_size)
        self.layers = nn.ModuleList([LlamaDecoderLayer_KIVI(config, i) for i in range(config.num_hidden_layers)])
        self.norm = LlamaRMSNorm(config.hidden_size, config.rms_norm_eps)


class KiviPast(tuple):
    """The per-layer `past_key_value` that forward() hands out while the cache lives in the pre-allocated KiviCache.
    It indexes like the reference's 9-tuple (models/llama_kivi.py:454-455): [8] / [-1] is kv_seq_len (what
    prepare_inputs_for_generation reads, :917) and costs nothing; the eight tensors are exported from the blocked cache
    on first access (a snapshot).  Passing it back to forward() continues on the fused path; it is valid for that as long
    as the cache has not moved on (one step per forward call, like the reference's functional tuples)."""

    def __new__(cls, cache, layer: int, kv_len: int):
        self = super().__new__(cls, ())
        self.cache, self.layer, self.kv_len, self._fields = cache, layer, kv_len, None
        return self

    def materialise(self):
        if self._fields is None:
            if self.cache.kv_len != self.kv_len:
                raise RuntimeError(f"stale KIVI cache view: it describes {self.kv_len} tokens, the cache now holds "
                                   f"{self.cache.kv_len} (export a view before decoding further if you need a snapshot)")
            self._fields = self.cache.export(self.layer)
        return self._fields

    def __len__(self):
        return 9

    def __getitem__(self, i):
        if isinstance(i, int) and i in (8, -1):
            return self.kv_len
        return self.materialise()[i]

    def __iter__(self):
        return iter(self.materialise())

    def __repr__(self):
        return f"KiviPast(layer={self.layer}, kv_seq_len={self.kv_len})"


class _Output(tuple):
    """What forward() returns when no transformers ModelOutput class is wanted: a (logits, past_key_values) tuple that
    also answers to the attribute names of CausalLMOutputWithPast."""
    __slots__ = ()
    loss = None
    logits = property(lambda self: self[0])
    past_key_values = property(lambda self: self[1])


def _additive_mask(attention_mask, q_len: int, total: int, dtype, device):
    """HF padding mask [B, total] (1 = attend) -> additive [B, 1, q_len, total] with the causal structure, or None
    when nothing is masked; a 4-D additive mask passes through (what the reference's hook receives, :364-372)."""
    if attention_mask is None:
        return None
    if attention_mask.dim() == 4:
        return attention_mask
    keep = attention_mask[:, None, None, :total].to(torch.bool)
    if q_len == 1 and bool(keep.all()):
        return None
    if q_len > 1:
        causal = torch.ones((q_len, total), dtype=torch.bool, device=device).tril(total - q_len)
        keep = keep & causal
    else:
        keep = keep.expand(-1, 1, 1, total)
    return torch.zeros(keep.shape, dtype=dtype, device=device).masked_fill(~keep, torch.finfo(dtype).min)


def _left_padding(attention_mask):
    """HF padding mask [B, n] (1 = real token) -> (pad [B], positions [B, n]), both int64 on the mask's device, or None when
    nothing is padded.  pad[b] counts the leading zeros of row b; positions are those of prepare_inputs_for_generation
    (cumsum - 1, padding at 1).  The fused cache path supports LEFT padding only: the zeros of every row must form a prefix.
    Right padding or holes raise NotImplementedError, a row without a real token ValueError."""
    if attention_mask is None:
        return None
    if attention_mask.dim() != 2:
        raise NotImplementedError("the fused cache path takes a 2-D HF padding mask [batch, tokens] with left padding")
    keep = attention_mask.to(torch.bool)
    if bool(keep.all()):
        return None
    if not bool(keep.any(-1).all()):
        raise ValueError("attention_mask has a row without any real token")
    m = keep.long()
    if not bool((m[:, 1:] >= m[:, :-1]).all()):
        raise NotImplementedError("the fused cache path supports left padding only (the zeros of every attention_mask row "
                                  "must form a prefix); right padding and holes are not supported")
    pad = m.shape[1] - m.sum(-1)
    positions = m.cumsum(-1) - 1
    positions.masked_fill_(m == 0, 1)
    return pad, positions


class LlamaForCausalLM_KIVI(nn.Module):
    """models/llama_kivi.py:785.  `forward` keeps the reference's contract (HF argument names, per-layer 9-tuples as
    past_key_values, fp32 logits, `prepare_inputs_for_generation`, `_reorder_cache`); `decode_step` / `generate` use
    the fused cache path (pre-allocated KiviCache, the step captured in a CUDA graph)."""

    def __init__(self, config):
        super().__init__()
        self.config = config
        self.vocab_size = config.vocab_size
        self.model = LlamaModel_KIVI(config)
        self.lm_head = nn.Linear(config.hidden_size, config.vocab_size, bias=False)
        self._rope = None
        self.cache: KiviCache | None = None
        self._graph = None
        self._graph_padded = False          # whether the captured step launches the padded attention (cache.seq_start set)
        self._fast = None
        self._dist_tokens = None            # [world * B] ids gathered inside the step (greedy sampling, world > 1)
        self._dist_in_graph = True
        self._exchange = None               # kivi_b200.dist.PeerTokenExchange: ids stored into the peers' buffers by the sampling kernel
        self._sampling_user = None          # the values given to set_sampling (generate's base values)
        self._sampling_cfg = None           # the values decode_step samples with (None: greedy decoding)
        self._sampling = None               # glue.SamplingParams: their device buffers, sized to the cache's batch

    # ------------------------------------------------------------------ HF-style construction
    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path, config=None, torch_dtype=torch.float16, device_map=None,
                        **unused):
        """Load a LOCAL Hugging Face Llama / Mistral checkpoint directory (config.json + *.safetensors or
        pytorch_model*.bin; there is no network here) into the KIVI model, as the reference's
        LlamaForCausalLM_KIVI.from_pretrained(config=...) does (example.py:22-28, mem_spd_test.py:24-31).  `config` is
        the user's config object carrying k_bits / v_bits / group_size / residual_length (models/llama_kivi.py:34-38);
        without one, config.json is read and the KIVI attributes default to K2V2 g32 R128."""
        import glob
        import json
        import os
        path = str(pretrained_model_name_or_path)
        if not os.path.isdir(path):
            raise FileNotFoundError(f"{path}: from_pretrained needs a local checkpoint directory (no network on this box)")
        if config is None:
            with open(os.path.join(path, "config.json")) as f:
                raw = json.load(f)
            config = SimpleNamespace(**raw)
        for name, dflt in (("k_bits", 2), ("v_bits", 2), ("group_size", 32), ("residual_length", 128), ("use_flash", True)):
            if not hasattr(config, name):
                setattr(config, name, dflt)
        model = cls(config)
        state = {}
        files = sorted(glob.glob(os.path.join(path, "*.safetensors")))
        if files:
            from safetensors.torch import load_file
            for fn in files:
                state.update(load_file(fn))
        else:
            for fn in sorted(glob.glob(os.path.join(path, "pytorch_model*.bin"))):
                state.update(torch.load(fn, map_location="cpu", weights_only=True))
        if not state:
            raise FileNotFoundError(f"{path}: no *.safetensors / pytorch_model*.bin weights found")
        if "lm_head.weight" not in state and getattr(config, "tie_word_embeddings", False):
            state["lm_head.weight"] = state["model.embed_tokens.weight"]
        state = {k: v for k, v in state.items() if not k.endswith("rotary_emb.inv_freq")}
        model.load_state_dict(state, strict=True)
        if torch_dtype is not None:
            model = model.to(torch_dtype)
        if device_map is not None:          # "auto" / "cuda" / {"": device}: one replica on the current GPU (dp, not pipeline)
            model = model.cuda()
        return model.eval()

    def get_input_embeddings(self):
        return self.model.embed_tokens

    def get_output_embeddings(self):
        return self.lm_head

    def _apply(self, fn, *args, **kwargs):
        # .to() / .half() / .cuda() re-create every parameter: the fused decode buffers and the captured graph would keep
        # pointing at the old storage
        self._fast, self._graph, self._rope = None, None, None
        return super()._apply(fn, *args, **kwargs)

    # ------------------------------------------------------------------ helpers
    def _tables(self, device):
        rows = getattr(self.config, "max_position_embeddings", 4096)
        if self.cache is not None:
            rows = max(rows, self.cache.max_tokens + 1)   # a cache longer than the config's context still has its rows
        if self._rope is None or self._rope[0].device != device or self._rope[0].shape[0] < rows:
            hd = self.config.hidden_size // self.config.num_attention_heads
            self._rope = _rope_tables(hd, rows, self.config.rope_theta, device)
        return self._rope

    def _run_layers(self, input_ids, positions, pasts, attention_mask=None):
        cos_t, sin_t = self._tables(input_ids.device)
        cos = cos_t.index_select(0, positions.reshape(-1)).view(positions.shape[0], 1, positions.shape[1], -1)
        sin = sin_t.index_select(0, positions.reshape(-1)).view(positions.shape[0], 1, positions.shape[1], -1)
        h = self.model.embed_tokens(input_ids)
        new_pasts = []
        for i, layer in enumerate(self.model.layers):
            h, past = layer(h, cos, sin, pasts[i] if pasts is not None else None, attention_mask)
            new_pasts.append(past)
        h = self.model.norm(h)
        return h, new_pasts

    # ------------------------------------------------------------------ reference-style forward (9-tuples)
    @torch.no_grad()
    def forward(self, input_ids=None, past_key_values=None, attention_mask=None, position_ids=None, use_cache=None,
                return_dict=None, **unused):
        """models/llama_kivi.py:815-905.  Returns logits [B, q_len, vocab] fp32 (:881) and past_key_values = per-layer
        9-tuples (:696-698, :911-916); prefill when past_key_values is None.  attention_mask: HF padding mask
        [B, kv_len] or an additive [B, 1, q_len, kv_len].  The result unpacks as (logits, past_key_values) and has the
        attributes of CausalLMOutputWithPast; with return_dict=True (or config.use_return_dict) it IS one."""
        B, q_len = input_ids.shape
        if past_key_values is not None and len(past_key_values) == 0:
            past_key_values = None
        start = 0 if past_key_values is None else past_key_values[0][-1]
        fused = self._fused_forward_ok(input_ids, past_key_values, attention_mask, position_ids, start)
        if fused:
            logits, pasts = self._forward_fused(input_ids, past_key_values, start)
        else:
            if past_key_values is not None and isinstance(past_key_values[0], KiviPast):
                past_key_values = [tuple(p.materialise()) for p in past_key_values]     # leave the fused path: plain 9-tuples
            if position_ids is None:
                position_ids = torch.arange(start, start + q_len, device=input_ids.device).unsqueeze(0).expand(B, -1)
            rows = self._tables(input_ids.device)[0].shape[0]
            if start + q_len > rows:            # the slow path's index_select would raise; say why
                raise ValueError(f"{start + q_len} positions exceed config.max_position_embeddings = {rows}")
            dtype = self.lm_head.weight.dtype
            mask = _additive_mask(attention_mask, q_len, start + q_len, dtype, input_ids.device)
            h, pasts = self._run_layers(input_ids, position_ids, past_key_values, mask)
            logits = self.lm_head(h).float()                                     # logits.float() (:881)
        if return_dict is None:
            return_dict = getattr(self.config, "use_return_dict", False)
        if return_dict:
            from transformers.modeling_outputs import CausalLMOutputWithPast
            return CausalLMOutputWithPast(loss=None, logits=logits, past_key_values=tuple(pasts))
        return _Output((logits, pasts))

    # ------------------------------------------------------------------ forward() on the fused cache path
    fused_forward = True        # False: forward() always uses the reference's own 9-tuples (torch.cat growth, per-op launches)

    def _fused_forward_ok(self, input_ids, past_key_values, attention_mask, position_ids, start):
        """forward() may run on the pre-allocated cache when nothing asks for what only the tuple path offers: CUDA fp16
        weights, equal-length sequences (no padding mask), default positions, and -- with a past -- one new token."""
        if not self.fused_forward or not input_ids.is_cuda or not self._fast_ok():
            return False
        B, q_len = input_ids.shape
        if attention_mask is not None and (attention_mask.dim() != 2 or not bool(attention_mask.to(torch.bool).all())):
            return False
        if position_ids is not None:
            exp = torch.arange(start, start + q_len, device=position_ids.device).unsqueeze(0).expand(B, -1)
            if position_ids.shape != exp.shape or not bool((position_ids == exp).all()):
                return False
        if past_key_values is None:
            return True
        if q_len != 1 or len(past_key_values) != len(self.model.layers):
            return False
        if isinstance(past_key_values[0], KiviPast):
            return all(isinstance(p, KiviPast) and p.cache is self.cache and p.kv_len == self.cache.kv_len
                       for p in past_key_values)
        return past_key_values[0][5] is not None and past_key_values[0][5].shape[0] == B      # plain 9-tuples: import once

    def _forward_fused(self, input_ids, past_key_values, start):
        B, q_len = input_ids.shape
        n_layers = len(self.model.layers)
        reserve = int(getattr(self.config, "kivi_cache_reserve", 1024))      # head-room allocated beyond the current length
        if past_key_values is None:                                          # prefill into the blocked cache
            if self.cache is None or self.cache.batch != B or self.cache.max_tokens < q_len + 1:
                self.init_cache(B, q_len + reserve)
            positions = torch.arange(q_len, device=input_ids.device).unsqueeze(0).expand(B, -1)
            h, _ = self._run_layers(input_ids, positions, [(self.cache, i) for i in range(n_layers)])
            self._pos.fill_(q_len)
            logits = self.lm_head(h).float()
        else:
            if not isinstance(past_key_values[0], KiviPast):                 # a cache grown elsewhere (reference hook): one re-layout
                self.import_cache(past_key_values, max_tokens=start + reserve)
            elif self.cache.kv_len + 1 > self.cache.max_tokens:              # out of room: re-allocate at twice the size
                tuples = [self.cache.export(i) for i in range(n_layers)]
                self.import_cache(tuples, max_tokens=2 * self.cache.max_tokens)
            logits = self.decode_step(input_ids).unsqueeze(1).clone()
        kv = self.cache.kv_len
        return logits, [KiviPast(self.cache, i, kv) for i in range(n_layers)]

    def prepare_inputs_for_generation(self, input_ids, past_key_values=None, attention_mask=None, inputs_embeds=None,
                                      **kwargs):
        """models/llama_kivi.py:908-948: feed only the tokens the cache has not seen (its length is the last element
        of a layer's tuple), positions from the padding mask."""
        if past_key_values is not None and len(past_key_values) == 0:
            past_key_values = None
        if past_key_values is not None:
            seen = past_key_values[0][-1]
            drop = seen if input_ids.shape[1] > seen else input_ids.shape[1] - 1
            input_ids = input_ids[:, drop:]
        position_ids = kwargs.get("position_ids")
        if attention_mask is not None and position_ids is None:
            position_ids = attention_mask.long().cumsum(-1) - 1
            position_ids.masked_fill_(attention_mask == 0, 1)
            if past_key_values:
                position_ids = position_ids[:, -input_ids.shape[1]:]
        return {"input_ids": input_ids, "position_ids": position_ids, "past_key_values": past_key_values,
                "use_cache": kwargs.get("use_cache"), "attention_mask": attention_mask}

    @staticmethod
    def _reorder_cache(past_key_values, beam_idx):
        """models/llama_kivi.py:950-957 (beam search): select batch rows of every tensor of every layer's tuple; the
        reference's version fails on the None entries and the trailing int of the 9-tuple -- they pass through here."""
        return tuple(tuple(t.index_select(0, beam_idx.to(t.device)) if torch.is_tensor(t) else t for t in layer_past)
                     for layer_past in past_key_values)

    # ------------------------------------------------------------------ fused cache path
    def init_cache(self, batch: int, max_tokens: int):
        cfg = self.config
        dev = self.lm_head.weight.device
        self.cache, self._graph = None, None                 # release the previous cache before the new one is allocated
        self.cache = KiviCache(cfg.num_hidden_layers, batch, cfg.num_attention_heads, cfg.num_key_value_heads,
                               cfg.hidden_size // cfg.num_attention_heads, cfg.k_bits, cfg.v_bits, cfg.group_size,
                               cfg.residual_length, max_tokens, device=dev,
                               overlap_prologue=True)       # the attention call follows the layer's RoPE kernel
        self._graph = None
        self._pos = torch.zeros((batch, 1), dtype=torch.long, device=dev)
        self._ids = torch.zeros((batch, 1), dtype=torch.long, device=dev)
        self._logits = torch.zeros((batch, cfg.vocab_size), dtype=torch.float32, device=dev)
        self.next_tokens = torch.zeros((batch,), dtype=torch.long, device=dev)   # the ids sampled by the step (in-graph)
        self._sampling = None
        self._tables(dev)                                    # rows for every position the cache can reach
        return self.cache

    def import_cache(self, past_key_values, max_tokens: int | None = None):
        """Continue on the fused path from the reference's per-layer 9-tuples (models/llama_kivi.py:454-455)."""
        seen = past_key_values[0][-1]
        B = past_key_values[0][5].shape[0]
        if self.cache is None or self.cache.batch != B or max(max_tokens or 0, seen + 1) > self.cache.max_tokens:
            self.init_cache(B, max(max_tokens or 0, seen + 1024))
        for i, past in enumerate(past_key_values):
            self.cache.import_tuple(i, past)
        self._pos.fill_(seen)
        return self.cache

    @torch.no_grad()
    def prefill(self, input_ids, attention_mask=None):
        """Run the prompt, fill the cache (models/llama_kivi.py:401-452), return last-position logits.
        attention_mask: None, or an HF padding mask [B, n] with LEFT padding (the zeros of every row form a prefix).  The
        prompt then runs with HF's positions and padding mask, and the decode steps mask the padding of every sequence
        (KiviCache.set_seq_start) and continue its positions from its number of real tokens."""
        assert self.cache is not None, "call init_cache() first"
        B, n = input_ids.shape
        if attention_mask is not None and tuple(attention_mask.shape) != (B, n):
            raise ValueError(f"attention_mask of shape {tuple(attention_mask.shape)} for input_ids of shape {(B, n)}")
        padding = _left_padding(attention_mask)
        pasts = [(self.cache, i) for i in range(len(self.model.layers))]
        if padding is None:
            positions = torch.arange(n, device=input_ids.device).unsqueeze(0).expand(B, -1)
            h, _ = self._run_layers(input_ids, positions, pasts)
            self._pos.fill_(n)
        else:
            pad, positions = padding
            mask = _additive_mask(attention_mask, n, n, self.lm_head.weight.dtype, input_ids.device)
            h, _ = self._run_layers(input_ids, positions.to(input_ids.device), pasts, mask)
            self._pos.copy_((n - pad).view(B, 1))
            self.cache.set_seq_start(pad)                    # after the layers: KiviCache.prefill switches padding off
        return self.lm_head(h[:, -1]).float()

    @torch.no_grad()
    def prefill_synthetic(self, n: int, seed: int = 0, seq_start=None):
        """Fill every layer's cache with n random K/V tokens (benchmarks: the prompt's attention itself is
        off the decode hot path; the cache contents are produced by the real prefill pack kernels).
        seq_start: None, or one int per sequence: its first real position (left padding, as prefill with a mask sets it)."""
        assert self.cache is not None
        c = self.cache
        gen = torch.Generator(device=c.device).manual_seed(seed)
        for l in range(c.n_layers):
            k = torch.randn((c.batch, c.num_kv_heads, n, c.head_dim), generator=gen, device=c.device, dtype=torch.float16)
            v = torch.randn((c.batch, c.num_kv_heads, n, c.head_dim), generator=gen, device=c.device, dtype=torch.float16)
            c.prefill(l, k, v)
        self._pos.fill_(n)
        if seq_start is not None:
            c.set_seq_start(seq_start)
            self._pos.copy_((n - c.seq_start.long().clamp(0, n)).view(c.batch, 1))

    def _step_body(self):
        if self._fast_ok():
            self._step_body_fast()
        else:
            pasts = [(self.cache, i) for i in range(len(self.model.layers))]
            h, _ = self._run_layers(self._ids, self._pos, pasts)
            self._logits.copy_(self.lm_head(h[:, 0]).float())
        self.cache_advance_device()
        self._pos.add_(1)
        # sampling inside the step (and inside its CUDA graph): the id of a sequence needs only that sequence's logits,
        # so with data-parallel replicas the exchange is the sampled ids, 8 B per sequence
        from . import glue
        if self._exchange is not None:
            self._exchange.step.add_(1)                      # the step number the peers' arrival counters are compared with
        # one kernel: argmax (or temperature / top-k / top-p draw) per sequence, the feed-back copy for the next step, and
        # (replicas) the ids stored straight into every peer's buffer over NVLink + arrival counters
        if self._sampling_cfg is None:
            glue.greedy_sample(self._logits, self.next_tokens, self._ids.view(-1), self._exchange)
        else:
            sp = self._sampling_params()
            sp.counter.add_(1)                               # a new uniform per step, also on graph replays
            glue.sample(self._logits, sp, self.next_tokens, self._ids.view(-1), self._exchange)
        if self._dist_tokens is not None and self._dist_in_graph:
            from . import dist as kdist
            kdist.gather_tokens(self.next_tokens, out=self._dist_tokens)

    def enable_token_allgather(self, world_size: int, in_graph: bool = True, mode: str = "nccl"):
        """Data-parallel replicas (kivi_b200.dist): every rank's sampled ids end up in `all_tokens` [world_size * B].
        mode "p2p": the sampling kernel itself stores the ids into every peer's symmetric buffer (PeerTokenExchange; one
        fused compute + collective kernel inside the step's CUDA graph).  mode "nccl": an NCCL all-gather of the ids, inside
        the graph (in_graph) or right after the replay.  Call before the first decode_step (the step is captured once)."""
        self._exchange, self._dist_tokens = None, None
        if world_size > 1 and mode == "p2p":
            from . import dist as kdist
            self._exchange = kdist.PeerTokenExchange(self.cache.batch, self.cache.device)
        elif world_size > 1:
            self._dist_tokens = torch.zeros(world_size * self.cache.batch, dtype=torch.long, device=self.cache.device)
        self._dist_in_graph = in_graph
        self._graph = None

    def set_sampling(self, temperature=1.0, top_k=0, top_p=1.0, seed: int | None = None):
        """Sample the steps of decode_step with temperature -> top-k -> top-p (transformers' warpers; kivi_sample_exchange_f32
        in include/kivi_b200.h); `set_sampling(None)` returns to greedy decoding.  Every value is one number or one per
        sequence: temperature 0 makes that sequence greedy, top_k 0 and top_p 1 switch the filter off.  seed=None draws one
        from torch's default generator (torch.manual_seed makes it reproducible).  Changing values is a device copy that
        the captured step sees; switching between greedy and sampling re-captures the step.  The draw counter restarts at 0."""
        self._sampling_user = None if temperature is None else dict(temperature=temperature, top_k=top_k, top_p=top_p,
                                                                       seed=seed)
        self._activate_sampling(self._sampling_user)

    def _activate_sampling(self, cfg):
        if cfg is None:
            if self._sampling_cfg is not None:
                self._graph = None
            self._sampling_cfg = None
            return
        cfg = dict(cfg)
        if cfg["seed"] is None:
            cfg["seed"] = int(torch.randint(0, 2 ** 63 - 1, (1,)).item())
        if self._sampling_cfg is None:
            self._graph = None
        self._sampling_cfg = cfg
        if self.cache is not None:
            self._sampling_params().set(counter=0, **cfg)

    def _sampling_params(self):
        """The device buffers of the sampling values, (re)made for the current cache batch and filled on creation."""
        from . import glue
        c = self.cache
        if self._sampling is None or self._sampling.batch != c.batch or self._sampling.temperature.device != c.device:
            import torch.distributed as tdist
            rank = tdist.get_rank() if tdist.is_available() and tdist.is_initialized() else 0
            self._sampling = glue.SamplingParams(c.batch, c.device, row_offset=rank * c.batch)   # rows of a global batch
            self._sampling.set(counter=0, **self._sampling_cfg)
            self._graph = None
        return self._sampling

    @property
    def all_tokens(self):
        if self._exchange is not None:
            return self._exchange.tokens()
        return self.next_tokens if self._dist_tokens is None else self._dist_tokens

    def _fast_ok(self):
        a = self.model.layers[0].self_attn
        return a.head_dim == 128 and a.q_proj.bias is None and self.lm_head.weight.dtype == torch.float16

    def _ensure_fast(self):
        """Fused q|k|v, o and gate|up weights in [in, out] layout + static activation buffers for the 9-launch-per-layer
        step.  At M = B rows cuBLAS streams the weights 9-13 % faster from this layout (tools/gemm_probe.py: q|k|v 27.6 vs
        31.8 us, o 15.4 vs 17.4 us, gate|up 42.0 vs 46.1 us; down is layout-neutral).  The fused buffers OWN the storage:
        the nn.Linear parameters become transposed views of them, so there is one copy of every weight (the reference's
        mem_spd_test reports peak memory) and load_state_dict / in-place edits reach the decode path."""
        if self._fast is not None and self._fast.B == self.cache.batch:
            return self._fast
        cfg, dev, B = self.config, self.cache.device, self.cache.batch
        H, Hkv, hid, inter = cfg.num_attention_heads, cfg.num_key_value_heads, cfg.hidden_size, cfg.intermediate_size
        f = self._fast if self._fast is not None else SimpleNamespace(wqkv=None)
        f.B = B
        if f.wqkv is None:
            def view_param(buf, lo, hi):
                return nn.Parameter(buf.t()[lo:hi], requires_grad=False)
            f.wqkv, f.wgu, f.wo = [], [], []
            for l in self.model.layers:
                a, m = l.self_attn, l.mlp
                nq, nk = a.q_proj.weight.shape[0], a.k_proj.weight.shape[0]
                w = torch.cat([a.q_proj.weight, a.k_proj.weight, a.v_proj.weight], 0).t().contiguous()
                a.q_proj.weight, a.k_proj.weight = view_param(w, 0, nq), view_param(w, nq, nq + nk)
                a.v_proj.weight = view_param(w, nq + nk, w.shape[1])
                f.wqkv.append(w)
                w = torch.cat([m.gate_proj.weight, m.up_proj.weight], 0).t().contiguous()
                m.gate_proj.weight, m.up_proj.weight = view_param(w, 0, inter), view_param(w, inter, 2 * inter)
                f.wgu.append(w)
                w = a.o_proj.weight.t().contiguous()
                a.o_proj.weight = view_param(w, 0, w.shape[1])
                f.wo.append(w)
        e = lambda *shape: torch.empty(shape, dtype=torch.float16, device=dev)  # noqa: E731
        f.res, f.h, f.o, f.d = e(B, hid), e(B, hid), e(B, hid), e(B, hid)
        f.qkv, f.q, f.k, f.v = e(B, (H + 2 * Hkv) * 128), e(B, H, 128), e(B, Hkv, 128), e(B, Hkv, 128)
        f.attn, f.gu, f.act = e(B, H, 128), e(B, 2 * inter), e(B, inter)
        f.logits16 = e(B, cfg.vocab_size)
        self._fast = f
        return f

    def _step_body_fast(self):
        """One decode step with 9 launches per layer: 4 cuBLAS GEMMs (q|k|v, o, gate|up, down), RoPE+split,
        fused KIVI attention, SiLU*mul and two residual-add+RMSNorm kernels."""
        from . import glue
        f = self._ensure_fast()
        cfg, cache = self.config, self.cache
        cos_t, sin_t = self._tables(cache.device)
        eps = cfg.rms_norm_eps
        layers = self.model.layers
        f.res.copy_(self.model.embed_tokens(self._ids)[:, 0])
        glue.add_rmsnorm(None, f.res, layers[0].input_layernorm.weight, f.h, eps)
        for i, l in enumerate(layers):
            torch.mm(f.h, f.wqkv[i], out=f.qkv)
            glue.rope_split(f.qkv, cos_t, sin_t, self._pos, f.q, f.k, f.v)
            cache.decode_attention(i, f.q, f.k, f.v, out=f.attn)
            torch.mm(f.attn.view(f.B, -1), f.wo[i], out=f.o)
            glue.add_rmsnorm(f.o, f.res, l.post_attention_layernorm.weight, f.h, eps)
            torch.mm(f.h, f.wgu[i], out=f.gu)
            glue.silu_mul(f.gu, f.act)
            torch.mm(f.act, l.mlp.down_proj.weight.t(), out=f.d)
            nxt = layers[i + 1].input_layernorm.weight if i + 1 < len(layers) else self.model.norm.weight
            glue.add_rmsnorm(f.d, f.res, nxt, f.h, eps)
        torch.mm(f.h, self.lm_head.weight.t(), out=f.logits16)
        self._logits.copy_(f.logits16)                                       # logits.float() (:881)

    def cache_advance_device(self):
        from . import _lib
        import ctypes
        with torch.cuda.device(self.cache.device):
            _lib.check(_lib.lib().kivi_cache_advance(ctypes.byref(self.cache._structs[0]),
                                                     _lib.stream_ptr(self.cache.device)), "kivi_cache_advance")

    @torch.no_grad()
    def decode_step(self, input_ids=None, use_graph: bool = True):
        """One decode step for the whole batch: input_ids [B, 1] (device) -> logits [B, vocab] fp32 (device,
        a static buffer); `next_tokens` [B] holds their argmax, or the ids drawn with set_sampling's values (and
        `all_tokens` every rank's, see enable_token_allgather).  The step (32 x [norm, qkv, rope, fused KIVI attention, o_proj, MLP], lm_head,
        cache advance, greedy argmax, token all-gather) is captured once in a CUDA graph and replayed."""
        assert self.cache is not None
        if self.cache.kv_len + 1 > self.cache.max_tokens:
            raise ValueError("KIVI cache capacity exceeded")
        if input_ids is not None:
            self._ids.copy_(input_ids.view(-1, 1))
        sp = self._sampling_params() if self._sampling_cfg is not None else None   # made before a capture, never inside
        padded = self.cache.seq_start is not None
        if self._graph is not None and self._graph_padded != padded:
            self._graph = None                               # the captured step launches the other attention entry
        if not use_graph:
            self._step_body()
        else:
            if self._graph is None:
                # warm-up on a side stream (cuBLAS workspaces, lazy module loading, NCCL channels), then capture
                state = self.cache.state.clone()
                pos, ids0 = self._pos.clone(), self._ids.clone()
                ctr = sp.counter.clone() if sp is not None else None
                s = torch.cuda.Stream()
                s.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(s):
                    self._step_body()
                torch.cuda.current_stream().wait_stream(s)
                torch.cuda.synchronize()
                # undo the warm-up step's effect on the lengths.  Everything it wrote lies BEYOND them -- the new token's
                # window slots (K slot r, the free slot of the V ring), a flushed K block past tk, the packed V token at
                # tv -- and is rewritten with the same bytes by the first replayed step.
                self.cache.state.copy_(state)
                self._pos.copy_(pos)
                self._ids.copy_(ids0)
                if sp is not None:
                    sp.counter.copy_(ctr)                                    # the warm-up step drew nothing for the caller
                from . import _lib
                n0 = _lib.launch_count()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._step_body()
                self.launches_per_step = _lib.launch_count() - n0            # libkivi_b200 launches replayed by every step
                # capture does not execute: state is still the pre-step state
                self._graph, self._graph_padded = g, padded
            self._graph.replay()
        if self._dist_tokens is not None and not self._dist_in_graph:
            from . import dist as kdist
            kdist.gather_tokens(self.next_tokens, out=self._dist_tokens)
        self.cache._mirror_advance()
        return self._logits

    @torch.no_grad()
    def generate(self, input_ids=None, max_new_tokens: int | None = None, use_graph: bool = True, attention_mask=None,
                 max_length: int | None = None, do_sample: bool = False, temperature: float | None = None,
                 top_k: int | None = None, top_p: float | None = None, seed: int | None = None, **unused):
        """Decoding on the fused path with the call shape of HF generate (`model.generate(**inputs, max_new_tokens=n)`,
        example.py:60-61, mem_spd_test.py:66): returns [B, prompt + new] ids.  do_sample=False: greedy (the model's decode
        steps return to greedy; set_sampling's values stay for the next do_sample=True).  do_sample=True:
        every token, the first one after the prompt included, is drawn inside the step by the sampling kernel with the
        values given to set_sampling, overridden by any of temperature / top_k / top_p / seed given here; values never
        given are transformers' defaults (1.0, 50, 1.0), a seed never given is drawn from torch's default generator, and
        the draw counter restarts at every call.  attention_mask: an HF padding mask with LEFT padding (prefill): the batch
        keeps one kv_seq_len, as the reference's cache does (:309, :455), and every sequence's padding is masked in every
        step; the padding stays on the left of the returned ids, as HF returns them."""
        if do_sample:
            if temperature is not None and not temperature > 0:
                raise ValueError(f"`temperature` (={temperature}) has to be a strictly positive float when sampling")
            cfg = dict(self._sampling_user or dict(temperature=1.0, top_k=50, top_p=1.0, seed=None))
            given = dict(temperature=temperature, top_k=top_k, top_p=top_p, seed=seed)
            cfg.update({k: v for k, v in given.items() if v is not None})
        else:
            self._activate_sampling(None)
        B, n = input_ids.shape
        _left_padding(attention_mask)                        # a mask the fused path cannot run raises before any work
        if max_new_tokens is None:
            if max_length is None:
                raise ValueError("generate() needs max_new_tokens or max_length")
            max_new_tokens = max_length - n
        if self.cache is None or self.cache.batch != B or self.cache.max_tokens < n + max_new_tokens:
            self.init_cache(B, n + max_new_tokens)
        logits = self.prefill(input_ids, attention_mask)
        out = [input_ids]
        if do_sample:
            self._activate_sampling(cfg)                     # counter 0: the first draw below uses counter 1
            sp = self._sampling_params()
            sp.counter.add_(1)
            from . import glue
            tok = glue.sample(logits.contiguous(), sp, torch.empty(B, dtype=torch.long, device=logits.device)).view(B, 1)
        else:
            tok = logits.argmax(-1, keepdim=True)
        for _ in range(max_new_tokens - 1):
            out.append(tok)
            self.decode_step(tok, use_graph=use_graph)
            tok = self.next_tokens.view(B, 1).clone()
        out.append(tok)
        return torch.cat(out, dim=1)


MistralForCausalLM_KIVI = LlamaForCausalLM_KIVI       # models/mistral_kivi.py:921 -- same hook; GQA is handled in-kernel
MistralFlashAttention_KIVI = LlamaFlashAttention_KIVI  # (no repeat_kv_quant copies, models/mistral_kivi.py:58-67)
