// kivi_decode.cu -- C-ABI entry of the decode attention; the kernels live in kivi_attn.cuh and are instantiated
// per (k_bits, v_bits) pair in kivi_attn_k{2,4}v{2,4}.cu (compiled in parallel).
#include <cstdlib>
#include "kivi_attn.cuh"

namespace kivi {
int attention_k2v2(AttnParams& p, int G, bool overlap_prologue, cudaStream_t st);
int attention_k4v4(AttnParams& p, int G, bool overlap_prologue, cudaStream_t st);
int attention_k2v4(AttnParams& p, int G, bool overlap_prologue, cudaStream_t st);
int attention_k4v2(AttnParams& p, int G, bool overlap_prologue, cudaStream_t st);
}

using namespace kivi;

// query heads of a KV head that share one unit's MMAs: from the cache geometry, or the explicit KIVI_CACHE_GQA_CHUNK
// field of cache->flags (the same struct sizes the workspace and launches, so both always agree)
static int gqa_chunk(int ratio, int flags) {
    int G = ratio % 4 == 0 ? 4 : (ratio % 2 == 0 ? 2 : 1);
    const int want = (flags >> KIVI_CACHE_GQA_CHUNK_SHIFT) & 7;
    if ((want == 1 || want == 2 || want == 4) && ratio % want == 0) G = want;
    return G;
}

extern "C" int64_t kivi_decode_workspace_bytes(const kivi_cache_t* cache, int max_kv_len)
{
    CacheDesc c;
    int rc = make_desc(cache, &c);
    if (rc) return rc;
    if (max_kv_len <= 0) return KIVI_ERR_SHAPE;
    const int ratio = c.H / c.Hkv, G = gqa_chunk(ratio, cache->flags);
    return carve_workspace(c, c.B * c.Hkv * (ratio / G), G, max_kv_len, nullptr, nullptr);
}

// the launch path of both entries: mask and seq_start are never both set
static int decode_attention(const kivi_cache_t* cache, const void* q, const void* k_new, const void* v_new,
                            const void* mask, const int32_t* seq_start, void* out, void* workspace, int64_t workspace_bytes,
                            void* dbg_logits, void* dbg_probs, int64_t dbg_stride, int max_kv_len, void* stream)
{
    AttnParams p;
    int rc = make_desc(cache, &p.c);
    if (rc) return rc;
    if (!q || !k_new || !v_new || !out || !workspace) return KIVI_ERR_NULL;
    if (max_kv_len <= 0) return KIVI_ERR_SHAPE;
    if (max_kv_len > p.c.k_cap_blocks * kBlockTokens) return KIVI_ERR_CAPACITY;
    if (reinterpret_cast<uintptr_t>(workspace) % 256 != 0) return KIVI_ERR_ALIGN;
    p.q = (const __half*)q; p.k_new = (const __half*)k_new; p.v_new = (const __half*)v_new; p.mask = (const __half*)mask;
    p.seq_start = seq_start;
    p.out = (__half*)out; p.dbg_logits = (__half*)dbg_logits; p.dbg_probs = (__half*)dbg_probs; p.dbg_stride = dbg_stride;
    const bool overlap = (cache->flags & KIVI_CACHE_OVERLAP_PROLOGUE) != 0;   // the q.K^T launch may overlap its predecessor
    const int ratio = p.c.H / p.c.Hkv;
    const int G = gqa_chunk(ratio, cache->flags);
    p.hchunks = ratio / G;
    p.n_units = p.c.B * p.c.Hkv * p.hchunks;
    p.max_kv_len = max_kv_len;
    const int64_t need = carve_workspace(p.c, p.n_units, G, max_kv_len, workspace, &p.w);
    if (need < 0) return (int)need;
    if (need > workspace_bytes) return KIVI_ERR_CAPACITY;
    cudaStream_t st = (cudaStream_t)stream;
    if (p.c.k_bits == 2 && p.c.v_bits == 2) return attention_k2v2(p, G, overlap, st);
    if (p.c.k_bits == 4 && p.c.v_bits == 4) return attention_k4v4(p, G, overlap, st);
    if (p.c.k_bits == 2 && p.c.v_bits == 4) return attention_k2v4(p, G, overlap, st);
    if (p.c.k_bits == 4 && p.c.v_bits == 2) return attention_k4v2(p, G, overlap, st);
    return KIVI_ERR_BITS;
}

extern "C" int kivi_decode_attention_f16(const kivi_cache_t* cache, const void* q, const void* k_new, const void* v_new,
                                         const void* mask, void* out, void* workspace, int64_t workspace_bytes,
                                         void* dbg_logits, void* dbg_probs, int64_t dbg_stride, int max_kv_len, void* stream)
{
    return decode_attention(cache, q, k_new, v_new, mask, nullptr, out, workspace, workspace_bytes, dbg_logits, dbg_probs,
                            dbg_stride, max_kv_len, stream);
}

extern "C" int kivi_decode_attention_padded_f16(const kivi_cache_t* cache, const void* q, const void* k_new, const void* v_new,
                                                const int32_t* seq_start, void* out, void* workspace, int64_t workspace_bytes,
                                                void* dbg_logits, void* dbg_probs, int64_t dbg_stride, int max_kv_len,
                                                void* stream)
{
    if (!seq_start) return KIVI_ERR_NULL;
    return decode_attention(cache, q, k_new, v_new, nullptr, seq_start, out, workspace, workspace_bytes, dbg_logits, dbg_probs,
                            dbg_stride, max_kv_len, stream);
}

// Test hook (tests/test_ranges_cpu.py): the work split of the decode kernels, evaluated on the host.  kernel 0 = q.K^T costs,
// 1 = p.V costs; out_lo receives (unit, item) of the first position of ranges 0 .. W (2 * (W + 1) ints, the last = the end);
// out_owner (may be NULL) receives owner(unit, item) for every position in order.  Returns W (or a negative error).
extern "C" int kivi_debug_range_split(int n_units, int n_b, int n_w, int w_cap, int kernel, int* out_lo, int* out_owner)
{
    if (n_units <= 0 || n_b < 0 || n_w < 0 || w_cap <= 0 || !out_lo) return KIVI_ERR_SHAPE;
    auto run = [&](auto rg) {
        for (int w = 0; w <= (int)rg.W; ++w) rg.lo(w, out_lo[2 * w], out_lo[2 * w + 1]);
        if (out_owner)
            for (int u = 0; u < n_units; ++u)
                for (int j = 0; j < rg.per_unit; ++j) out_owner[(long long)u * rg.per_unit + j] = rg.owner(u, j);
        return (int)rg.W;
    };
    if (kernel == 0) { Ranges<CostQK> rg; rg.init(n_units, n_b, n_w, w_cap); return run(rg); }
    Ranges<CostSV> rg; rg.init(n_units, n_b, n_w, w_cap);
    return run(rg);
}

#if KIVI_TIMELINE
#include <vector>
namespace kivi {
int timeline_k2v2(unsigned long long*); int timeline_k2v4(unsigned long long*);
int timeline_k4v2(unsigned long long*); int timeline_k4v4(unsigned long long*);
}
// tuning builds only (tools/timeline.py): the per-warp timestamps of the last attention call, [2][4096][8]
extern "C" int kivi_debug_timeline(unsigned long long* host_out)
{
    const size_t n = 2 * 4096 * 8;
    std::vector<unsigned long long> tmp(n);
    for (size_t i = 0; i < n; ++i) host_out[i] = 0;
    int (*fetch[4])(unsigned long long*) = {timeline_k2v2, timeline_k2v4, timeline_k4v2, timeline_k4v4};
    for (auto f : fetch) {
        const int rc = f(tmp.data());
        if (rc) return rc;
        for (size_t i = 0; i < n; ++i) if (tmp[i] > host_out[i]) host_out[i] = tmp[i];   // timestamps: the latest writer wins
    }
    return 0;
}
#endif
