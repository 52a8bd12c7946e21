"""Oracle of sampled decoding (kivi_sample_exchange_f32, include/kivi_b200.h): a numpy Philox4x32-10 and a float64
restatement of temperature -> top-k -> top-p -> draw.

The kernel sums its masses in fp32 exp / fixed point, so a row whose top-p boundary (S_>(v) against p*Z1) or draw boundary
(running mass against u*Z_K) lies within `rel` * Z of a decision may legitimately go either way: `acceptable_ids` returns,
per row, every id the rule gives when those boundaries move by up to `rel` relative to Z.  The temperature division and the
top-k threshold are exact (fp32 l / T is bit-identical here and on the GPU), and greedy rows have one answer.
"""
from __future__ import annotations

import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)


def philox4x32_10(counter, key):
    """counter uint32 [..., 4], key uint32 [..., 2] -> uint32 [..., 4] (Random123's philox4x32, 10 rounds)."""
    c = [np.asarray(counter, dtype=np.uint64)[..., i] for i in range(4)]
    k0 = np.asarray(key, dtype=np.uint64)[..., 0]
    k1 = np.asarray(key, dtype=np.uint64)[..., 1]
    for _ in range(10):
        p0, p1 = _M0 * c[0], _M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK]
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return np.stack(c, -1).astype(np.uint32)


def uniforms(seed: int, counter: int, rows):
    """u = ((r0 >> 8) + 0.5) * 2^-24 for the given global rows (float64, exact)."""
    rows = np.asarray(rows, dtype=np.int64)
    seed, counter = int(seed) & (2 ** 64 - 1), int(counter) & (2 ** 64 - 1)
    ctr = np.zeros(rows.shape + (4,), dtype=np.uint32)
    ctr[..., 0], ctr[..., 1], ctr[..., 2] = counter & 0xFFFFFFFF, counter >> 32, rows.astype(np.uint32)
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint32), rows.shape + (2,))
    r0 = philox4x32_10(ctr, key)[..., 0]
    return ((r0 >> np.uint32(8)).astype(np.float64) + 0.5) * 2.0 ** -24


def scaled(row, T):
    """x = fp32(l / T), NaN -> -inf, -0 -> +0 (the kernel's step 1 for a sampled row)."""
    x = (np.asarray(row, dtype=np.float32) / np.float32(T)).astype(np.float32)
    x[np.isnan(x)] = -np.inf
    x[x == 0] = 0.0
    return x


def masses(x):
    """e = exp(x - max) in float64; at an infinite maximum the tokens equal to it share the mass."""
    mx = x.max()
    with np.errstate(invalid="ignore"):
        d = x.astype(np.float64) - np.float64(mx)
    d[np.isnan(d)] = np.where(x[np.isnan(d)] == mx, 0.0, -np.inf)
    return np.exp(d)


def topk_survivors(x, k):
    V = x.shape[0]
    if k <= 0 or k >= V:
        return np.ones(V, dtype=bool)
    return x >= np.sort(x)[V - k]


def _strictly_greater_mass(x, e, surv):
    """S_>(v) for every v: mass of the survivors with a strictly larger x."""
    xs, es = x[surv], e[surv]
    vals, inv = np.unique(xs, return_inverse=True)             # ascending distinct values
    per = np.bincount(inv, weights=es, minlength=len(vals))
    above = np.concatenate([np.cumsum(per[::-1])[::-1][1:], [0.0]])   # mass of the values strictly above each value
    idx = np.searchsorted(vals, x)
    idx = np.clip(idx, 0, len(vals) - 1)
    return above[idx]


def kept_mask(row, T, k, p):
    """The nominal kept set of a sampled row (steps 1-3)."""
    x = scaled(row, T)
    e = masses(x)
    surv = topk_survivors(x, k)
    if p >= 1:
        return surv
    sg = _strictly_greater_mass(x, e, surv)
    return surv & ((sg < p * e[surv].sum()) | (x == x.max()))


def _draw_band(e, kept, u, rel):
    m = np.where(kept, e, 0.0)
    cum = np.cumsum(m)
    zk = cum[-1]
    last = int(np.flatnonzero(kept)[-1])
    if not zk > 0:
        return last, {last}
    t = u * zk
    hit = np.flatnonzero(cum > t)
    pick = int(hit[0]) if hit.size else last
    d = rel * zk
    band = np.flatnonzero((m > 0) & (cum > t - d) & (cum - m <= t + d))
    return pick, set(int(i) for i in band) | {pick}


def acceptable_ids(logits, temperature, top_k, top_p, seed, counter, row_offset=0, rel=1e-5):
    """(picks [B] int64, list of sets of acceptable ids) for fp32 logits [B, V] and per-row parameters."""
    logits = np.asarray(logits, dtype=np.float32)
    B, V = logits.shape
    T = np.broadcast_to(np.asarray(temperature, dtype=np.float32), (B,))
    K = np.broadcast_to(np.asarray(top_k, dtype=np.int64), (B,))
    P = np.broadcast_to(np.asarray(top_p, dtype=np.float32), (B,))
    us = uniforms(seed, counter, row_offset + np.arange(B))
    picks, sets = np.zeros(B, dtype=np.int64), []
    for b in range(B):
        row = logits[b]
        if not T[b] > 0:                                   # greedy row: first NaN, else the first maximum
            nan = np.flatnonzero(np.isnan(row))
            i = int(nan[0]) if nan.size else int(np.argmax(row))
            picks[b] = i
            sets.append({i})
            continue
        x = scaled(row, T[b])
        e = masses(x)
        surv = topk_survivors(x, int(K[b]))
        p = float(P[b])
        if p >= 1:
            variants, nominal = [surv], 0
        else:
            sg = _strictly_greater_mass(x, e, surv)
            z1 = e[surv].sum()
            thr, d = np.float64(p) * z1, rel * z1
            top = x == x.max()
            lo = surv & ((sg < thr - d) | top)
            border = np.unique(sg[surv & ~lo & (sg < thr + d)])   # groups whose fate lies within the band, by S_>
            variants = [lo | (surv & np.isin(sg, border[:j])) for j in range(len(border) + 1)]
            nominal = int(np.sum(border < thr))
        acc = set()
        for j, kept in enumerate(variants):
            pick, band = _draw_band(e, kept, us[b], rel)
            acc |= band
            if j == nominal:
                picks[b] = pick
        sets.append(acc)
    return picks, sets
