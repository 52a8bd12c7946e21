/*
 * kivi_b200.h -- C ABI of libkivi_b200.so, the B200-native (sm_100a) implementation of the
 * KIVI decode hot path: 2/4-bit asymmetric pack of new K/V tokens and the batched dequant-GEMVs
 * q.K^T and softmax.V over the packed cache (+ fp16 residual window).
 *
 * This is the drop-in boundary.  Each entry point replaces one interface of the reference
 * (jy-yuan/KIVI @ 876b4d2); the reference-side binding a maintainer would add is shown in
 * INTEGRATION.md.  Rules common to all entry points:
 *   - plain C types only: device pointers, sizes, strides, a stream handle.  No torch types.
 *   - the CALLER owns every buffer, outputs included; nothing is allocated, nothing is freed.
 *   - asynchronous: work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = the
 *     legacy default stream) and the call returns immediately.  No global state, re-entrant,
 *     CUDA-graph capturable.  The device is the current device of the calling thread and must
 *     own the pointers (the Python shim wraps calls in torch.cuda.device(tensor.device)).
 *   - return 0 on success, a negative KIVI_ERR_* for argument errors (nothing was enqueued),
 *     or a positive cudaError_t from the launch.  Never throws.
 *   - fp16 data are IEEE binary16 (`__half` bits); packed codes are little-endian in the
 *     32-bit word: element i of a word sits at bit i*bits (quant/new_pack.py:148-153).
 */
#ifndef KIVI_B200_H
#define KIVI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KIVI_OK              0
#define KIVI_ERR_BITS       -1   /* bits not in the supported set                         */
#define KIVI_ERR_SHAPE      -2   /* a dimension / divisibility requirement is violated    */
#define KIVI_ERR_GQA        -3   /* nh % nh_kv != 0 or nh_kv <= 0                         */
#define KIVI_ERR_GROUP      -4   /* unsupported group_size                                */
#define KIVI_ERR_ALIGN      -5   /* pointer / stride alignment requirement violated       */
#define KIVI_ERR_NULL       -6   /* required pointer is NULL                              */
#define KIVI_ERR_LAYOUT     -7   /* unknown layout id                                     */
#define KIVI_ERR_CAPACITY   -8   /* cache capacity exceeded                               */
#define KIVI_ERR_UNSUPPORTED -9  /* valid in the reference, not implemented by this build */

#define KIVI_LAYOUT_REFERENCE 0  /* qB [U, K, N/fpi], scales/zeros [U, K, N/g]  (quant/matmul.py:189-191) */
#define KIVI_LAYOUT_KERNEL    1  /* qB [U, N/fpi, K], scales/zeros [U, N/g, K]  (quant/csrc/gemv_cuda.cu:255-259) */

/* Library identification. */
int         kivi_version(void);
const char* kivi_error_string(int code);
/* Number of kernel launches this library has enqueued since load (bench.py's gpu_launches). */
uint64_t    kivi_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Pack: asymmetric min/max quantisation along the LAST dim in groups of `group_size`,
 * OR-packed into int32 words.
 * Replaces triton_quantize_and_pack_along_last_dim(data, group_size, bit),
 *   quant/new_pack.py:217-252 (Triton _minmax_along_last_dim :158-177, ATen chain :238-242,
 *   Triton _pack_along_last_dim :132-154) -- one fused kernel instead of >= 9 launches.
 * Bit-exact on codes, scale and mn (fp16 rounding chain of SURVEY 8 a1); degenerate group
 * (mx == mn) -> code 0, scale 0.
 *   x     [rows, T]       fp16, contiguous
 *   code  [rows, T/fpi]   int32   (fpi = 32/bits)
 *   scale [rows, T/g]     fp16
 *   mn    [rows, T/g]     fp16
 * Requires bits in {2,4,8}, T % group_size == 0 (quant/new_pack.py:222), T % fpi == 0.
 * ------------------------------------------------------------------------------------------ */
int kivi_pack_lastdim_f16(const void* x, int64_t rows, int64_t T, int group_size, int bits,
                          void* code, void* scale, void* mn, void* stream);

/* ------------------------------------------------------------------------------------------
 * Batched "outer-dim" dequant-GEMV:  C[u_q, n] = sum_k A[u_q, k] * (scale*code + zero)[u_kv, k, n],
 * u_kv = u_q / (nh / nh_kv); groups and packing run along n.  fp32 accumulate, fp16 store.
 * Replaces
 *   layout KIVI_LAYOUT_KERNEL   : kivi_gemv.gemv_forward_cuda_outer_dim(in, kernel, scales, zeros,
 *                                 bit, group_size, nh, nh_kv), quant/csrc/gemv_cuda.h:12-20,
 *                                 quant/csrc/gemv_cuda.cu:511-557 (+ kernels :265-427);
 *   layout KIVI_LAYOUT_REFERENCE: the whole of cuda_bmm_fA_qB_outer, quant/matmul.py:178-219,
 *                                 WITHOUT its three transpose().contiguous() copies (:205,213-214).
 *   A      fp16, U_q = B*nh rows of K elements; row u at A + u*a_stride (elements), unit stride in k
 *   qB     int32, U_kv = B*nh_kv units, unit u at qB + u*qb_unit_stride (words);
 *            REFERENCE: word (k, n/fpi) at k*qb_row_stride + n/fpi
 *            KERNEL   : word (n/fpi, k) at (n/fpi)*qb_row_stride + k
 *   scales/zeros fp16, unit u at + u*sz_unit_stride (elements);
 *            REFERENCE: (k, n/g) at k*sz_row_stride + n/g ;  KERNEL: (n/g, k) at (n/g)*sz_row_stride + k
 *   C      fp16 [U_q, N] contiguous
 * Requires bits in {2,4} (8 also accepted on KIVI_LAYOUT_REFERENCE, the Triton surface
 * quant/matmul.py:112-175), nh % nh_kv == 0, group_size % fpi == 0, N % group_size == 0.
 * (M, the number of query rows per head, is 1: the reference kernel ignores blockIdx.z,
 *  quant/csrc/gemv_cuda.cu:538.)
 * ------------------------------------------------------------------------------------------ */
int kivi_bgemv_outer_f16(const void* A, int64_t a_stride,
                         const void* qB, int64_t qb_unit_stride, int64_t qb_row_stride,
                         const void* scales, const void* zeros, int64_t sz_unit_stride, int64_t sz_row_stride,
                         void* C, int B, int nh, int nh_kv, int K, int N,
                         int bits, int group_size, int layout, void* stream);

/* ------------------------------------------------------------------------------------------
 * Inner-dim (AWQ-style) GEMV: out[b, oc] = sum_ic in[b, ic] * (scale*code + zero)[oc, ic/g],
 * packing and groups along ic.
 * Replaces kivi_gemv.gemv_forward_cuda(in, kernel, scales, zeros, bit, group_size),
 *   quant/csrc/gemv_cuda.h:4-10, quant/csrc/gemv_cuda.cu:201-246 (kernels :60-184; 4-bit only,
 *   scales/zeros rows padded to sf_w = g64: ceil(ceil(IC/64/8)/2)*2*8, g128: ceil(IC/128/8)*8),
 *   and the Triton gemv_fwd / gemv_kernel_g64 of quant/gemv.py:16-90 (any bit, sf_w = IC/g).
 *   in [Bn, IC] fp16; kernel [OC, IC/fpi] int32; scales/zeros [OC, sf_w] fp16; out [Bn, OC] fp16.
 * The reference silently returns uninitialised memory for group sizes other than 64/128
 * (:227-245); here every group_size % fpi == 0 is computed.  IC % fpi == 0.
 * ------------------------------------------------------------------------------------------ */
int kivi_gemv_inner_f16(const void* in, const void* kernel, const void* scales, const void* zeros,
                        void* out, int Bn, int IC, int OC, int bits, int group_size, int64_t sf_w,
                        void* stream);

/* ------------------------------------------------------------------------------------------
 * Unpack + dequantise along the last dim in fp16: out = fp16(fp16(code * scale) + mn).
 * Replaces unpack_and_dequant_vcache / unpack_and_dequant_kcache (quant/new_pack.py:51-83),
 * the reference's own test oracle for the pack path.  bits in {2,4,8}.
 *   code [rows, T/fpi] int32; scale, mn [rows, T/g] fp16; out [rows, T] fp16.
 * ------------------------------------------------------------------------------------------ */
int kivi_unpack_dequant_lastdim_f16(const void* code, const void* scale, const void* mn,
                                    int64_t rows, int64_t T, int group_size, int bits,
                                    void* out, void* stream);

/* ==========================================================================================
 * Pre-allocated KIVI cache + fused decode attention (the hot path of
 * LlamaFlashAttention_KIVI.forward, models/llama_kivi.py:314-399, and its Mistral twin).
 *
 * The reference keeps a per-layer 9-tuple of tensors that it regrows with torch.cat every step
 * (:350-352, :391-395, :454-455).  Here the caller allocates fixed buffers once (sizes from
 * kivi_cache_sizes) and describes one LAYER's cache with a kivi_cache_t; `state` is a device
 * int32[8] shared by all layers of a model {tk, r, tv, L, vhead, kv_len, -, -}: tk = tokens in the
 * packed K store, r = tokens in the fp16 K window, tv = tokens in the packed V store, L = tokens in
 * the fp16 V window (ring buffer starting at vhead).  All sequences of the batch have the same
 * length, as in the reference (one kv_seq_len per cache, :309, :455); a left-padded batch keeps
 * that shared length and gives each sequence its first real position instead
 * (kivi_decode_attention_padded_f16).
 * head_dim is 128 (every model the reference ships); group_size in {32,64,128};
 * residual_length % group_size == 0 (:344), residual_length in {32, 64, 128, 256}.
 * ========================================================================================== */
/* kivi_cache_t.flags.  KIVI_CACHE_OVERLAP_PROLOGUE: the caller promises that the kernel enqueued on the stream
 * directly before kivi_decode_attention_f16 never writes this cache (stores, windows) or its `state` -- true inside a
 * decoder layer, where that kernel produces q / k_new / v_new.  The q.K^T launch then starts under programmatic
 * dependent launch: it reads `state` and its first K blocks while that kernel drains, and waits for it only before
 * touching q / k_new.  Without the flag the q.K^T kernel is an ordinary launch (safe directly after
 * kivi_cache_advance / kivi_cache_prefill_f16 / a previous attention call on the same cache). */
#define KIVI_CACHE_OVERLAP_PROLOGUE 1
/* Bits 4..6 of kivi_cache_t.flags: how many query heads of a KV head share one work unit of the decode attention
 * (their MMAs and every packed byte): 0 = chosen from the geometry (4 if nh/nh_kv % 4 == 0, else 2, else 1), or an
 * explicit 1 / 2 / 4 dividing nh/nh_kv.  kivi_decode_workspace_bytes and kivi_decode_attention_f16 must see the same value. */
#define KIVI_CACHE_GQA_CHUNK_SHIFT 4
#define KIVI_CACHE_GQA_CHUNK(g)    ((g) << KIVI_CACHE_GQA_CHUNK_SHIFT)

typedef struct kivi_cache {
    int32_t batch, num_heads, num_kv_heads, head_dim;
    int32_t k_bits, v_bits, group_size, residual_length;
    int32_t k_cap_blocks;   /* capacity of the K store in 128-token blocks   (kivi_cache_sizes out[0]) */
    int32_t v_cap_blocks;   /* capacity of the V store in 128-token blocks   (out[1]) */
    int32_t v_res_cap;      /* slots of the fp16 V ring buffer               (out[2]) */
    int32_t flags;          /* KIVI_CACHE_* bits, 0 = none */
    void* k_store;          /* out[3] bytes */
    void* v_store;          /* out[4] bytes */
    void* k_res;            /* out[5] bytes */
    void* v_res;            /* out[6] bytes */
    void* state;            /* device int32[8], shared by the layers of one model */
} kivi_cache_t;

/* Buffer sizes for a cache that can hold max_tokens tokens per sequence: out[0..2] = capacities
 * (k_cap_blocks, v_cap_blocks, v_res_cap), out[3..6] = bytes of k_store, v_store, k_res, v_res.
 * Both stores are sequences of 128 x 128 "inner x outer" blocks (K: channel x token, V: token x channel;
 * quantisation groups along the outer dim) whose codes are laid out as mma.sync A-operand fragments and
 * whose scales / zeros are laid out as the B-fragment builders read them: kivi_b200/csrc/kivi_decode.cuh. */
int kivi_cache_sizes(int batch, int num_kv_heads, int k_bits, int v_bits, int group_size,
                     int residual_length, int max_tokens, int64_t* out);

/* Prefill: split + quantise the prompt's K/V exactly as models/llama_kivi.py:425-452 and set `state`.
 *   k, v [B, Hkv, n, 128] fp16 contiguous (K after RoPE).  K: the first n - n%R tokens (all n if
 *   R | n, none if n < R) are quantised per channel in groups of g tokens straight into the blocked
 *   store (fused transpose + quantise); V: the first n - R tokens per token in groups of g channels. */
int kivi_cache_prefill_f16(const kivi_cache_t* cache, const void* k, const void* v, int n, void* stream);

/* Bytes of the scratch workspace kivi_decode_attention_f16 needs for this cache geometry and contexts of up to
 * max_kv_len tokens (negative: KIVI_ERR_*).  The caller allocates it once, ZERO-INITIALISED (it holds arrival
 * counters that every call leaves at zero), 256-B aligned; one workspace can serve all layers of a model when
 * the layers run on one stream. */
int64_t kivi_decode_workspace_bytes(const kivi_cache_t* cache, int max_kv_len);

/* One decode step of attention for one layer (models/llama_kivi.py:314-399):
 *   logits = [ q.Kq^T (dequantise in register) | q.K_full^T | q.k_new ]   each rounded to fp16 (:324-337)
 *   s      = fp16(logits * (1/sqrt(128))) (+ mask, max with finfo.min)     (:339, :369-372)
 *   p      = fp16(softmax_fp32(s))                                          (:375)
 *   out    = fp16( fp16(p[:tv].Vq) + fp16(p[tv:].[V_full; v_new]) )         (:382-384)
 * then, per unit, the cache data movement of :343-356 / :386-399: k_new joins the fp16 K window or,
 * when that completes R tokens, the window is quantised into the K store; v_new joins the fp16 V
 * ring and, once it holds more than R tokens, its oldest token is quantised into the V store.
 * `state` is READ ONLY here; call kivi_cache_advance once per step after the last layer.
 *   q [B, H, 128], k_new / v_new [B, Hkv, 128], out [B, H, 128]  fp16 contiguous
 *   mask: NULL or additive fp16 [B, kv_len + 1] (broadcast over heads, :364-372).  Its row stride grows with
 *   every step, so a captured graph cannot reuse one mask buffer: left padding goes through
 *   kivi_decode_attention_padded_f16 below
 *   workspace / workspace_bytes: see kivi_decode_workspace_bytes (scaled logits rows, per-block softmax
 *   statistics, partial output records, arrival counters); no bound on the context length
 *   dbg_logits / dbg_probs: NULL or fp16 [B, H, dbg_stride] receiving s and p (tests)
 *   max_kv_len: the value the workspace was sized with (>= kv_len + 1).
 * Two launches on `stream`, no CTA barrier in either: every warp of a persistent grid (one 16-warp CTA per SM) is an
 * autonomous worker that owns one contiguous range of the (unit, 128-token block) sequence and streams its packed
 * blocks HBM -> shared memory with cp.async.bulk (TMA) into private mbarrier stages.  (1) q.K^T: a warp writes the
 * fp16 logits of its blocks and one (max, sum exp) pair per unit it touches.  (2) p.V (programmatic dependent launch
 * on (1)): a warp normalises its logits slices with the unit's combined statistics, accumulates, and writes one
 * partial record per unit; the last arriver of a unit adds the records in fixed order, rounds, writes `out` and
 * updates the cache.  The contraction of a packed block runs on mma.sync (codes as exact fp16 denormals x exact
 * hi/lo split of x*scale, fp32 accumulate); the query heads of a KV head share the MMAs (GQA).
 * Launch (1) reads `state` and its first K blocks at once: it is an ordinary launch unless cache->flags has
 * KIVI_CACHE_OVERLAP_PROLOGUE (see there). */
int kivi_decode_attention_f16(const kivi_cache_t* cache, const void* q, const void* k_new, const void* v_new,
                              const void* mask, void* out, void* workspace, int64_t workspace_bytes,
                              void* dbg_logits, void* dbg_probs, int64_t dbg_stride, int max_kv_len, void* stream);

/* The same step for a LEFT-PADDED batch (HF left padding + padding attention_mask, models/llama_kivi.py:364-372), with one
 * int per sequence instead of a mask row:
 *   seq_start: device int32 [B], required.  Positions 0 .. seq_start[b] - 1 of sequence b are padding; negative values
 *   count as 0.  The new token (position kv_len) is never padding, so no row is ever fully masked.
 * A padding position's scaled logit becomes what kivi_decode_attention_f16 gives for the mask value finfo(fp16).min
 * (-65504), so probabilities and outputs are bit-identical to that call with the equivalent mask.  seq_start is read on
 * the device by every call: a captured graph sees the values the caller copies into the same buffer before a replay.
 * Only the packed K blocks that overlap the padding take the predicated epilogue.  The cache update is unchanged:
 * padding tokens are quantised together with the real ones, as in the reference. */
int kivi_decode_attention_padded_f16(const kivi_cache_t* cache, const void* q, const void* k_new, const void* v_new,
                                     const int32_t* seq_start, void* out, void* workspace, int64_t workspace_bytes,
                                     void* dbg_logits, void* dbg_probs, int64_t dbg_stride, int max_kv_len, void* stream);

/* Test hook: the (unit, item) work split of the two decode kernels evaluated on the host (kernel 0 = q.K^T, 1 = p.V cost
 * model); a unit has n_b packed blocks, n_w window items and the new token.  out_lo: 2 * (W + 1) ints, (unit, item) of the first
 * position of every range and of the end; out_owner: NULL or one int per position.  Returns the number of ranges W. */
int kivi_debug_range_split(int n_units, int n_b, int n_w, int w_cap, int kernel, int* out_lo, int* out_owner);

/* Advance `state` by one token (the bookkeeping of :343-356, :386-399); once per step, all layers. */
int kivi_cache_advance(const kivi_cache_t* cache, void* stream);

/* Copy the 8 words of `state` to host memory (synchronises `stream`).  state[6] is an error word that the decode kernels
 * set instead of touching memory when the device-side lengths exceed what the call declared (max_kv_len, window
 * capacities): KIVI_STATE_ERR_CAPACITY.  kivi_cache_prefill_f16 / kivi_cache_import_f16 clear it. */
#define KIVI_STATE_ERR_CAPACITY 1
int kivi_cache_read_state(const kivi_cache_t* cache, int32_t* host_state8, void* stream);

/* Copy the cache out in the reference's 9-tuple layout (models/llama_kivi.py:454-455); lengths are
 * passed by the host (it mirrors `state`).  k_code [U,128,tk/fpi] i32, k_scale/k_mn [U,128,tk/g],
 * k_full [U,r,128], v_code [U,tv,128/fpi] i32, v_scale/v_mn [U,tv,128/g], v_full [U,L,128]. */
int kivi_cache_export_f16(const kivi_cache_t* cache, int tk, int r, int tv, int L, int vhead,
                          void* k_code, void* k_scale, void* k_mn, void* k_full,
                          void* v_code, void* v_scale, void* v_mn, void* v_full, void* stream);

/* The inverse of kivi_cache_export_f16: load one layer's cache from the reference's 9-tuple (the object a model that
 * ran on the reference's hook holds, models/llama_kivi.py:454-455) and set `state` = {tk, r, tv, L, 0, tk + r}.
 * Same operand shapes as the export; tk % residual_length == 0, r < residual_length, L <= residual_length,
 * tk + r == tv + L (both count the tokens seen).  Pointers of empty parts (tk == 0, r == 0, tv == 0) may be NULL. */
int kivi_cache_import_f16(const kivi_cache_t* cache, int tk, int r, int tv, int L,
                          const void* k_code, const void* k_scale, const void* k_mn, const void* k_full,
                          const void* v_code, const void* v_scale, const void* v_mn, const void* v_full, void* stream);

/* ------------------------------------------------------------------------------------------
 * Glue kernels of the decode step around the hot path (not part of the KIVI operators; they
 * replace ~16 ATen elementwise launches per layer per step in kivi_b200/llama_kivi.py).  fp16 I/O,
 * arithmetic of the HF Llama modules the reference forks: every fp16 op rounds to fp16.
 *   kivi_add_rmsnorm_f16 : residual += x (x may be NULL); out = weight * fp16(residual * rsqrt(mean(residual^2)+eps))
 *   kivi_rope_split_f16  : qkv [B,(H+2Hkv)*128] -> q [B,H,128], k [B,Hkv,128] (rotary at position pos[b], int64,
 *                          clamped to the table_rows rows of the cos / sin tables [table_rows, 128]), v
 *   kivi_silu_mul_f16    : gate_up [rows, 2*I] -> out [rows, I] = fp16(silu(gate)) * up
 * ------------------------------------------------------------------------------------------ */
int kivi_add_rmsnorm_f16(const void* x, void* residual, const void* weight, void* out,
                         int rows, int hidden, float eps, void* stream);
int kivi_rope_split_f16(const void* qkv, const void* cos_table, const void* sin_table, const void* pos,
                        void* q, void* k, void* v, int batch, int num_heads, int num_kv_heads, int table_rows,
                        void* stream);
int kivi_silu_mul_f16(const void* gate_up, void* out, int rows, int intermediate, void* stream);

/* Greedy sampling fused with its collective (the only exchange of the data-parallel decode, SURVEY 8e; the reference has
 * none).  next_local[b] = argmax_v logits[b, v] (first index among equal maxima, as torch.argmax; logits fp32 [batch, vocab],
 * models/llama_kivi.py:881); ids_feedback (may be NULL) receives the same ids (the next step's input buffer).
 * peer_buffers: NULL (one GPU), or a DEVICE array of `world` pointers, entry p = rank p's exchange buffer -- one symmetric
 * allocation per rank (peer-mapped over NVLink / NVSwitch), laid out as int64 tokens[2][world * batch] followed by
 * uint64 arrived[world], zero-initialised.  The kernel stores its ids into slot [step & 1][rank * batch + b] of EVERY rank's
 * buffer with plain peer stores, releases arrived[rank] on every peer, and waits (bounded, *err = 1 on time-out) until the
 * ids of all ranks for this step have arrived in its own buffer.  `step` is a device int32 the caller increments before each
 * call (the same on all ranks); all calls are CUDA-graph capturable. */
int kivi_greedy_sample_exchange_f32(const void* logits, int batch, int vocab, void* next_local, void* ids_feedback,
                                    const void* peer_buffers, int rank, int world, const void* step, void* err, void* stream);

/* Sampled decoding fused with the same exchange (temperature -> top-k -> top-p -> one draw; the order and definitions of
 * transformers' TemperatureLogitsWarper, TopKLogitsWarper, TopPLogitsWarper).  Per row b of logits fp32 [batch, vocab], with
 * T = temperature[b], k = top_k[b], p = top_p[b]:
 *   1. x_v = fp32(l_v / T) (IEEE division, as `scores / temperature`).  T <= 0: a GREEDY row, the argmax with the rule of
 *      kivi_greedy_sample_exchange_f32 (greedy and sampled rows may share a batch).  For sampled rows a NaN x counts as -inf.
 *   2. top-k (off when k <= 0 or k >= vocab): keep x_v >= x_(k), the k-th largest value; all ties at the threshold stay.
 *   3. top-p (off when p >= 1) over the top-k survivors, with e_v = exp(x_v - max x) and Z1 = sum e: keep v iff S_>(v) < p*Z1,
 *      S_>(v) = mass of the survivors with a strictly larger x (HF: drop where the ascending cumulative mass <= 1 - p;
 *      restated without a sort, so ties share one fate).  The maximum is always kept.
 *   4. draw: u = ((r0 >> 8) + 0.5) * 2^-24, r0 = word 0 of Philox4x32-10 with key (seed lo, seed hi) and counter
 *      (counter lo, counter hi, row_offset + b, 0).  The id is the smallest kept v (index order) whose running sum of e over
 *      the kept tokens exceeds u * Z_K, Z_K = the total of that sum; the last kept token if none does.
 * The masses are summed in 2^-40 fixed point, so every sum is exact and order-free: the ids are a pure function of (seed,
 * counter, row_offset + b, the logits row) -- the same in eager and graph mode, for any batch split across ranks, and from
 * run to run.  A row holding NaN or +-inf still yields an id in [0, vocab) (at an infinite maximum the tokens equal to it
 * share the mass).  vocab <= 262144; one cluster of up to 8 CTAs per row, the row held in shared memory.
 * next_local / ids_feedback / peer_buffers / rank / world / step / err: exactly as kivi_greedy_sample_exchange_f32. */
typedef struct kivi_sampling {
    const float*    temperature;  /* device [batch]; <= 0: greedy row                       */
    const int32_t*  top_k;        /* device [batch]; <= 0 or >= vocab: off                  */
    const float*    top_p;        /* device [batch]; >= 1: off                              */
    const uint64_t* seed;         /* device, 1 word                                         */
    const int64_t*  counter;      /* device, 1 word; the caller increments it before a call */
    int32_t         row_offset;   /* global index of row 0 (rank * batch)                   */
} kivi_sampling_t;
int kivi_sample_exchange_f32(const void* logits, int batch, int vocab, const kivi_sampling_t* s,
                             void* next_local, void* ids_feedback, const void* peer_buffers,
                             int rank, int world, const void* step, void* err, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* KIVI_B200_H */
