// kivi_model.cu -- small fused glue kernels of the decode step around the hot path (sm_100a):
// residual-add + RMSNorm, RoPE + q/k/v split, SiLU*mul.  They replace ~16 ATen elementwise launches per
// layer per step with 4; arithmetic follows the HF Llama modules the reference forks
// (models/llama_kivi.py star-imports transformers.models.llama): every fp16 op rounds to fp16.
#include "kivi_common.cuh"

namespace kivi {

// residual (fp16, in/out) += x;  out = weight * fp16( residual * rsqrt(mean(residual^2) + eps) )
// (LlamaRMSNorm.forward: fp32 statistics, cast to fp16, then multiply by the fp16 weight)
// One CTA per row, every thread keeps its 8-element slices in registers between the two passes.
template <bool ADD>
__global__ void __launch_bounds__(512)
add_rmsnorm_kernel(const __half* __restrict__ x, __half* __restrict__ residual, const __half* __restrict__ w,
                   __half* __restrict__ out, int hidden, float eps)
{
    constexpr int kMaxIter = 4;                          // hidden <= 4 * 512 * 8 = 16384
    __shared__ float red[16];
    const int row = blockIdx.x;
    __half* r = residual + (int64_t)row * hidden;
    const int nvec = hidden / 8;
    uint4 v[kMaxIter];
    float ss = 0.f;
    #pragma unroll
    for (int it = 0; it < kMaxIter; ++it) {
        const int i = threadIdx.x + it * 512;
        if (i < nvec) {
            uint4 u = *reinterpret_cast<const uint4*>(r + i * 8);
            __half2* h = reinterpret_cast<__half2*>(&u);
            if (ADD) {
                const uint4 xv = __ldg(reinterpret_cast<const uint4*>(x + (int64_t)row * hidden) + i);
                const __half2* xh = reinterpret_cast<const __half2*>(&xv);
                #pragma unroll
                for (int e = 0; e < 4; ++e) h[e] = __hadd2_rn(h[e], xh[e]);
                *reinterpret_cast<uint4*>(r + i * 8) = u;
            }
            #pragma unroll
            for (int e = 0; e < 4; ++e) { const float2 f = __half22float2(h[e]); ss = fmaf(f.x, f.x, fmaf(f.y, f.y, ss)); }
            v[it] = u;
        }
    }
    ss = warp_sum(ss);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    float tot = 0.f;
    #pragma unroll
    for (int i = 0; i < 16; ++i) tot += red[i];
    const float rs = rsqrtf(tot / (float)hidden + eps);
    #pragma unroll
    for (int it = 0; it < kMaxIter; ++it) {
        const int i = threadIdx.x + it * 512;
        if (i < nvec) {
            const __half2* h = reinterpret_cast<const __half2*>(&v[it]);
            const uint4 wv = __ldg(reinterpret_cast<const uint4*>(w) + i);
            const __half2* wh = reinterpret_cast<const __half2*>(&wv);
            uint4 o;
            __half2* oh = reinterpret_cast<__half2*>(&o);
            #pragma unroll
            for (int e = 0; e < 4; ++e) {
                const float2 f = __half22float2(h[e]);
                oh[e] = __hmul2_rn(wh[e], __floats2half2_rn(f.x * rs, f.y * rs));
            }
            *reinterpret_cast<uint4*>(out + (int64_t)row * hidden + i * 8) = o;
        }
    }
}

// qkv [B, (H + 2*Hkv) * 128] -> q [B,H,128], k [B,Hkv,128] (both rotated), v [B,Hkv,128]
// apply_rotary_pos_emb: x*cos + rotate_half(x)*sin, each op rounded to fp16; cos/sin rows = position pos[b]
__global__ void __launch_bounds__(64)
rope_split_kernel(const __half* __restrict__ qkv, const __half* __restrict__ cos_t, const __half* __restrict__ sin_t,
                  const long long* __restrict__ pos, __half* __restrict__ q, __half* __restrict__ k, __half* __restrict__ v,
                  int H, int Hkv, int table_rows)
{
    constexpr int D = 128;
    // the q.K^T kernel that follows is launched with programmatic serialization: let it set up and start streaming K blocks
    // while this kernel runs (it waits for our completion before it reads q / k / v)
    asm volatile("griddepcontrol.launch_dependents;");
    const int b = blockIdx.y, head = blockIdx.x, i = threadIdx.x;            // i < 64: pair (i, i + 64)
    const __half* src = qkv + ((int64_t)b * (H + 2 * Hkv) + head) * D;
    if (head >= H + Hkv) {                                                   // v: plain copy
        __half* dst = v + ((int64_t)b * Hkv + head - H - Hkv) * D;
        dst[i] = src[i]; dst[i + 64] = src[i + 64];
        return;
    }
    long long p = pos[b];
    p = p < 0 ? 0 : (p >= table_rows ? table_rows - 1 : p);                  // never read outside the tables (the host checks the range)
    const __half c0 = cos_t[p * D + i], c1 = cos_t[p * D + i + 64];
    const __half s0 = sin_t[p * D + i], s1 = sin_t[p * D + i + 64];
    const __half x0 = src[i], x1 = src[i + 64];
    __half* dst = head < H ? q + ((int64_t)b * H + head) * D : k + ((int64_t)b * Hkv + head - H) * D;
    dst[i] = __hadd_rn(__hmul_rn(x0, c0), __hmul_rn(__hneg(x1), s0));       // rotate_half: (-x2, x1)
    dst[i + 64] = __hadd_rn(__hmul_rn(x1, c1), __hmul_rn(x0, s1));
}

// gu [rows, 2*I] (gate | up) -> out [rows, I] = fp16(silu(gate)) * up
__global__ void __launch_bounds__(256)
silu_mul_kernel(const __half* __restrict__ gu, __half* __restrict__ out, int I)
{
    const int row = blockIdx.y;
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (i >= I) return;
    const float2 g = __half22float2(*reinterpret_cast<const __half2*>(gu + (int64_t)row * 2 * I + i));
    const __half2 u = *reinterpret_cast<const __half2*>(gu + (int64_t)row * 2 * I + I + i);
    const __half2 a = __floats2half2_rn(g.x / (1.f + expf(-g.x)), g.y / (1.f + expf(-g.y)));
    *reinterpret_cast<__half2*>(out + (int64_t)row * I + i) = __hmul2_rn(a, u);
}

// ------------------------------------------------------------------------------------------------
// Greedy sampling fused with its collective.  One block per sequence: argmax over the vocabulary (first index among equal
// maxima, like torch.argmax), then thread 0 stores the id into this rank's slot of EVERY rank's token buffer -- plain stores
// to peer memory over NVLink / NVSwitch (the buffers are one symmetric allocation, torch.distributed._symmetric_memory) --
// and releases a per-rank arrival counter on every peer.  Block 0 then waits (bounded) until all ranks' ids of this step have
// arrived here.  Argmax is local to a sequence, so the data-parallel replicas exchange 8 bytes per sequence and nothing of
// the next step depends on the exchange: no rank ever blocks another one's critical path.  The buffer layout, the stores
// and the bounded wait are exchange_publish / exchange_wait (kivi_common.cuh), shared with the sampling kernel.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
greedy_exchange_kernel(const float* __restrict__ logits, int V, long long* __restrict__ next_local, long long* __restrict__ ids_feedback,
                       long long* const* __restrict__ peer, int B, int rank, int world, const int* __restrict__ step_ptr, int* __restrict__ err)
{
    __shared__ float smax[8];
    __shared__ int sidx[8];
    const int b = blockIdx.x, tid = threadIdx.x;
    const TokenExchange x{peer, B, rank, world, step_ptr, err};
    const float* row = logits + (long long)b * V;
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int i = tid; i < V; i += 256) {
        const float v = row[i];
        if (argmax_takes(best, bi, v, i)) { best = v; bi = i; }             // a NaN wins, like torch.argmax
    }
    warp_argmax(best, bi);
    if ((tid & 31) == 0) { smax[tid >> 5] = best; sidx[tid >> 5] = bi; }
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < 8; ++w)
            if (argmax_takes(best, bi, smax[w], sidx[w])) { best = smax[w]; bi = sidx[w]; }
        exchange_publish(bi, b, next_local, ids_feedback, x);
    }
    if (b == 0) exchange_wait(x, tid);                                       // all ranks' ids of this step are here before the kernel ends
}

}  // namespace kivi

using namespace kivi;

extern "C" int kivi_greedy_sample_exchange_f32(const void* logits, int batch, int vocab, void* next_local, void* ids_feedback,
                                               const void* peer_buffers, int rank, int world, const void* step, void* err,
                                               void* stream)
{
    if (!logits || !next_local) return KIVI_ERR_NULL;
    if (batch <= 0 || vocab <= 0) return KIVI_ERR_SHAPE;
    if (peer_buffers && (!step || !err || world < 1 || rank < 0 || rank >= world || world > 256)) return KIVI_ERR_SHAPE;
    greedy_exchange_kernel<<<batch, 256, 0, (cudaStream_t)stream>>>(
        (const float*)logits, vocab, (long long*)next_local, (long long*)ids_feedback, (long long* const*)peer_buffers,
        batch, rank, world, (const int*)step, (int*)err);
    return post_launch();
}

extern "C" int kivi_add_rmsnorm_f16(const void* x, void* residual, const void* weight, void* out,
                                    int rows, int hidden, float eps, void* stream)
{
    if (!residual || !weight || !out) return KIVI_ERR_NULL;
    if (rows < 0 || hidden <= 0 || hidden % 8 != 0 || hidden > 16384) return KIVI_ERR_SHAPE;
    if (rows == 0) return KIVI_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (x) add_rmsnorm_kernel<true><<<rows, 512, 0, st>>>((const __half*)x, (__half*)residual,
                                                                            (const __half*)weight, (__half*)out, hidden, eps);
    else   add_rmsnorm_kernel<false><<<rows, 512, 0, st>>>(nullptr, (__half*)residual,
                                                                             (const __half*)weight, (__half*)out, hidden, eps);
    return post_launch();
}

extern "C" int kivi_rope_split_f16(const void* qkv, const void* cos_table, const void* sin_table, const void* pos,
                                   void* q, void* k, void* v, int batch, int num_heads, int num_kv_heads, int table_rows,
                                   void* stream)
{
    if (!qkv || !cos_table || !sin_table || !pos || !q || !k || !v) return KIVI_ERR_NULL;
    if (batch <= 0 || num_heads <= 0 || num_kv_heads <= 0 || batch > 65535 || table_rows <= 0) return KIVI_ERR_SHAPE;
    rope_split_kernel<<<dim3(num_heads + 2 * num_kv_heads, batch), 64, 0, (cudaStream_t)stream>>>(
        (const __half*)qkv, (const __half*)cos_table, (const __half*)sin_table, (const long long*)pos,
        (__half*)q, (__half*)k, (__half*)v, num_heads, num_kv_heads, table_rows);
    return post_launch();
}

extern "C" int kivi_silu_mul_f16(const void* gate_up, void* out, int rows, int intermediate, void* stream)
{
    if (!gate_up || !out) return KIVI_ERR_NULL;
    if (rows <= 0 || intermediate <= 0 || intermediate % 2 != 0 || rows > 65535) return KIVI_ERR_SHAPE;
    silu_mul_kernel<<<dim3(cdiv(intermediate / 2, 256), rows), 256, 0, (cudaStream_t)stream>>>(
        (const __half*)gate_up, (__half*)out, intermediate);
    return post_launch();
}
