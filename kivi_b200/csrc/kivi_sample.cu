// kivi_sample.cu -- sampled decoding (temperature -> top-k -> top-p -> one draw) fused with the token exchange (sm_100a).
//
// One thread-block cluster per row of the fp32 logits [B, V]: CTA r of the cluster loads the slice [r*L, (r+1)*L) of the row
// into shared memory ONCE, and every later pass reads it from there:
//   1. x = fp32(l / T) (IEEE division), max of the row (cluster merge through distributed shared memory)
//   2. top-k: radix select (4 x 8-bit digits) of the k-th largest order-preserving uint32 key of x
//   3. top-p: a mass-weighted radix select over the top-k survivors of the smallest key K with  S_>(K) < p * Z1
//   4. draw: the smallest kept index whose running mass (index order) exceeds u * Z_K
// The masses e = exp(x - max) are summed as 2^-40 fixed-point integers: every sum is exact, so the result does not depend
// on the order of the atomics or on the cluster split -- the ids are a pure function of (seed, counter, global row, row).
// The per-digit histograms of all CTAs of a cluster are merged through DSMEM; every CTA computes the same decisions.
// Rows with T <= 0 take the argmax with the order of the greedy kernel (kivi_model.cu).
#include <cooperative_groups.h>

#include "kivi_common.cuh"

namespace cg = cooperative_groups;

namespace kivi {
namespace smp {

constexpr int kThreads = 256;                          // == number of digit bins: thread t owns bin 255 - t in the merges
constexpr int kWarps = kThreads / 32;
constexpr int kMaxCluster = 8;                         // portable cluster size
constexpr int kMaxSlice = 32768;                       // floats of one CTA's slice (128 KB of shared memory)
constexpr int kMinSlice = 1024;                        // smaller rows use fewer CTAs
constexpr int kMaxVocab = kMaxCluster * kMaxSlice;
constexpr float kMassScale = 1099511627776.f;          // 2^40: e in [0, 1] -> integer mass

typedef unsigned long long u64;

// order-preserving key: a < b  <=>  key(a) < key(b) for non-NaN floats (-0 was canonicalised to +0 before)
__device__ __forceinline__ uint32_t order_key(float x) {
    const uint32_t u = __float_as_uint(x);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// e = exp(x - max) as a fixed-point integer.  x == max == +-inf (inf - inf) gives e = 1: the tokens at an infinite maximum
// share the mass (all of it for +inf; a row of only -inf is uniform).
__device__ __forceinline__ u64 mass(float x, float mx) {
    float d = x - mx;
    if (d != d) d = (x == mx) ? 0.f : -INFINITY;
    return __float2ull_rn(expf(d) * kMassScale);
}

// Philox4x32-10 (Salmon et al., SC'11; the Random123 / cuRAND generator), word 0 of the output block
__device__ __forceinline__ uint32_t philox4x32_10_w0(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    #pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t lo0 = 0xD2511F53u * c0, hi0 = __umulhi(0xD2511F53u, c0);
        const uint32_t lo1 = 0xCD9E8D57u * c2, hi1 = __umulhi(0xCD9E8D57u, c2);
        c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return c0;
}

struct Params {
    const float* logits;
    int V, L;                                          // row length, slice length per CTA
    const float* temperature;
    const int32_t* top_k;
    const float* top_p;
    const u64* seed;
    const long long* counter;
    int row_offset;
    long long* next_local;
    long long* ids_feedback;
    TokenExchange x;
};

// Merge bin (255 - t) of the histograms `buf` of every CTA of the cluster into `v` and scan it: incl = sum over the bins
// >= 255 - t.  Call after the cluster barrier that completes the histograms.
__device__ __forceinline__ void merge_scan(const cg::cluster_group& cl, u64* buf, int S, u64* wsum, u64& v, u64& incl) {
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    v = 0;
    for (int r = 0; r < S; ++r) v += cl.map_shared_rank(buf, r)[255 - t];
    incl = v;
    #pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u64 n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    u64 off = 0;
    for (int i = 0; i < w; ++i) off += wsum[i];
    incl += off;
    __syncthreads();                                   // wsum is free again
}

__global__ void __launch_bounds__(kThreads, 1)
sample_exchange_kernel(const Params p)
{
    extern __shared__ float xs[];                      // this CTA's slice: x = l / T
    __shared__ u64 hist[2][256];                       // per-digit counts / masses, double-buffered by pass parity
    __shared__ u64 wsum[kWarps];
    __shared__ u64 wtot[kWarps];                       // kept mass of each warp's segment (draw)
    __shared__ int wlast[kWarps];
    __shared__ float wmax[kWarps];
    __shared__ int widx[kWarps];
    __shared__ float cta_f;                            // published to the cluster: max (sampled) / best value (greedy)
    __shared__ int cta_i;                              //                            last kept index / best index
    __shared__ u64 cta_u;                              //                            kept mass of the slice
    __shared__ uint32_t s_prefix;
    __shared__ u64 s_acc;
    __shared__ int s_best;

    cg::cluster_group cl = cg::this_cluster();
    const int S = (int)cl.num_blocks(), crank = (int)cl.block_rank();
    const int b = blockIdx.y, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lo = crank * p.L;
    const int n = max(0, min(p.V, lo + p.L) - lo);
    const float* row = p.logits + (long long)b * p.V + lo;
    const float T = p.temperature[b];

    if (!(T > 0.f)) {                                  // ---- greedy row: argmax, first index among equal maxima, NaN wins
        float best = -INFINITY;
        int bi = 0x7fffffff;
        for (int i = tid; i < n; i += kThreads) {
            const float v = row[i];
            if (argmax_takes(best, bi, v, lo + i)) { best = v; bi = lo + i; }
        }
        warp_argmax(best, bi);
        if (lane == 0) { wmax[warp] = best; widx[warp] = bi; }
        __syncthreads();
        if (tid == 0) {
            for (int w = 1; w < kWarps; ++w)
                if (argmax_takes(best, bi, wmax[w], widx[w])) { best = wmax[w]; bi = widx[w]; }
            cta_f = best; cta_i = bi;
        }
        cl.sync();
        if (crank == 0 && tid == 0) {
            for (int r = 1; r < S; ++r) {
                const float ov = *cl.map_shared_rank(&cta_f, r);
                const int oi = *cl.map_shared_rank(&cta_i, r);
                if (argmax_takes(best, bi, ov, oi)) { best = ov; bi = oi; }
            }
            exchange_publish(bi < p.V ? bi : 0, b, p.next_local, p.ids_feedback, p.x);
        }
        cl.sync();                                     // the remote reads are done before any CTA exits
        if (b == 0 && crank == 0) exchange_wait(p.x, tid);
        return;
    }

    // ---- 1. load x = fp32(l / T) into shared memory (NaN -> -inf, -0 -> +0), max of the row
    float mx = -INFINITY;
    for (int i0 = tid; i0 < n; i0 += 4 * kThreads) {
        float v[4];
        #pragma unroll
        for (int j = 0; j < 4; ++j) { const int i = i0 + j * kThreads; v[j] = i < n ? row[i] : 0.f; }
        #pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int i = i0 + j * kThreads;
            if (i < n) {
                float x = __fdiv_rn(v[j], T);
                x = (x != x) ? -INFINITY : (x == 0.f ? 0.f : x);
                xs[i] = x;
                mx = fmaxf(mx, x);
            }
        }
    }
    #pragma unroll
    for (int o = 16; o >= 1; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) wmax[warp] = mx;
    __syncthreads();
    if (tid == 0) {
        for (int w = 1; w < kWarps; ++w) mx = fmaxf(mx, wmax[w]);
        cta_f = mx;
    }
    cl.sync();
    mx = -INFINITY;
    for (int r = 0; r < S; ++r) mx = fmaxf(mx, *cl.map_shared_rank(&cta_f, r));

    int pass = 0;
    // ---- 2. top-k: the k-th largest key Kk; every key >= Kk survives (all ties at the threshold)
    const int k = p.top_k[b];
    uint32_t Kk = 0;
    if (k > 0 && k < p.V) {
        uint32_t prefix = 0;
        u64 krem = (u64)k;
        for (int level = 0; level < 4; ++level, ++pass) {
            u64* buf = hist[pass & 1];
            buf[tid] = 0;
            __syncthreads();
            const int shift = 24 - 8 * level;
            const uint32_t hmask = level ? (0xffffffffu << (32 - 8 * level)) : 0u;
            for (int i = tid; i < n; i += kThreads) {
                const uint32_t key = order_key(xs[i]);
                if ((key & hmask) == prefix) atomicAdd(&buf[(key >> shift) & 255u], 1ull);
            }
            cl.sync();
            u64 v, incl;
            merge_scan(cl, buf, S, wsum, v, incl);
            if (incl - v < krem && krem <= incl) { s_prefix = prefix | ((uint32_t)(255 - tid) << shift); s_acc = krem - (incl - v); }
            __syncthreads();
            prefix = s_prefix;
            krem = s_acc;
        }
        Kk = prefix;
    }

    // ---- 3. top-p over the survivors: the smallest key Kp whose strictly-larger survivor mass is < p * Z1
    const float tp = p.top_p[b];
    uint32_t Kp = 0;
    if (tp < 1.f) {
        uint32_t prefix = 0;
        u64 above = 0;                                 // survivor mass above the current prefix range
        double thr = 0.0;
        for (int level = 0; level < 4; ++level, ++pass) {
            u64* buf = hist[pass & 1];
            buf[tid] = 0;
            if (tid == 0) s_best = -1;
            __syncthreads();
            const int shift = 24 - 8 * level;
            const uint32_t hmask = level ? (0xffffffffu << (32 - 8 * level)) : 0u;
            for (int i = tid; i < n; i += kThreads) {
                const float x = xs[i];
                const uint32_t key = order_key(x);
                if (key >= Kk && (key & hmask) == prefix) {
                    const u64 m = mass(x, mx);
                    if (m) atomicAdd(&buf[(key >> shift) & 255u], m);
                }
            }
            cl.sync();
            u64 v, incl;
            merge_scan(cl, buf, S, wsum, v, incl);
            if (level == 0) {
                if (tid == kThreads - 1) s_acc = incl;   // Z1
                __syncthreads();
                thr = (double)tp * (double)s_acc;
            }
            if ((double)(above + incl - v) < thr) atomicMax(&s_best, tid);
            __syncthreads();
            const int tb = s_best;
            if (tb < 0) { Kp = order_key(mx); break; }   // p <= 0 or a degenerate row: keep the maximum only
            if (tid == tb) { s_prefix = prefix | ((uint32_t)(255 - tb) << shift); s_acc = above + incl - v; }
            __syncthreads();
            prefix = s_prefix;
            above = s_acc;
            Kp = prefix;
        }
    }
    const uint32_t Kthr = max(Kk, Kp);

    // ---- 4. draw: kept mass per warp segment (index order), then the crossing of u * Z_K
    const int seg = cdiv(cdiv(max(n, 1), kWarps), 32) * 32;
    const int s0 = warp * seg, s1 = min(n, s0 + seg);
    u64 tot = 0;
    int last = -1;
    for (int i = s0 + lane; i < s1; i += 32) {
        const float x = xs[i];
        if (order_key(x) >= Kthr) { tot += mass(x, mx); last = i; }
    }
    #pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        tot += __shfl_xor_sync(0xffffffffu, tot, o);
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    }
    if (lane == 0) { wtot[warp] = tot; wlast[warp] = last; }
    __syncthreads();
    if (tid == 0) {
        u64 t = 0;
        int l = -1;
        for (int w = 0; w < kWarps; ++w) { t += wtot[w]; l = max(l, wlast[w]); }
        cta_u = t;
        cta_i = l < 0 ? -1 : lo + l;
    }
    cl.sync();
    u64 before = 0, zk = 0;
    int glast = -1;
    for (int r = 0; r < S; ++r) {
        const u64 t = *cl.map_shared_rank(&cta_u, r);
        if (r < crank) before += t;
        zk += t;
        glast = max(glast, *cl.map_shared_rank(&cta_i, r));
    }
    // u = (q + 0.5) 2^-24 with q = r0 >> 8; the id is the first kept v with running mass S_v > u Z_K, i.e. (S_v integer)
    // S_v > floor((2q + 1) Z_K / 2^25)
    const long long ctr = *p.counter;
    const u64 seed = *p.seed;
    const uint32_t r0 = philox4x32_10_w0((uint32_t)ctr, (uint32_t)((unsigned long long)ctr >> 32), (uint32_t)(p.row_offset + b), 0u,
                                         (uint32_t)seed, (uint32_t)(seed >> 32));
    const u64 a = 2ull * (r0 >> 8) + 1ull;
    const u64 plo = a * zk, phi = __umul64hi(a, zk);
    const u64 target = (phi << 39) | (plo >> 25);
    if (zk == 0) {                                     // nothing has mass (degenerate row): the last kept token
        if (crank == 0 && tid == 0) exchange_publish(glast >= 0 && glast < p.V ? glast : 0, b, p.next_local, p.ids_feedback, p.x);
    } else if (before <= target && target < before + cta_u) {
        u64 run = before;
        int w = 0;
        while (w < kWarps - 1 && run + wtot[w] <= target) run += wtot[w++];
        if (warp == w) {
            const int e0 = w * seg, e1 = min(n, e0 + seg);
            for (int i0 = e0; i0 < e1; i0 += 32) {
                const int i = i0 + lane;
                u64 m = 0;
                if (i < e1) { const float x = xs[i]; if (order_key(x) >= Kthr) m = mass(x, mx); }
                u64 incl = m;
                #pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const u64 t = __shfl_up_sync(0xffffffffu, incl, o);
                    if (lane >= o) incl += t;
                }
                const unsigned hit = __ballot_sync(0xffffffffu, run + incl > target);
                if (hit) {
                    if (lane == __ffs(hit) - 1) exchange_publish(lo + i, b, p.next_local, p.ids_feedback, p.x);
                    break;
                }
                run += __shfl_sync(0xffffffffu, incl, 31);
            }
        }
    }
    cl.sync();                                         // the remote reads are done before any CTA exits
    if (b == 0 && crank == 0) exchange_wait(p.x, tid);
}

}  // namespace smp
}  // namespace kivi

using namespace kivi;

extern "C" int kivi_sample_exchange_f32(const void* logits, int batch, int vocab, const kivi_sampling_t* s,
                                        void* next_local, void* ids_feedback, const void* peer_buffers,
                                        int rank, int world, const void* step, void* err, void* stream)
{
    using namespace kivi::smp;
    if (!logits || !s || !next_local) return KIVI_ERR_NULL;
    if (!s->temperature || !s->top_k || !s->top_p || !s->seed || !s->counter) return KIVI_ERR_NULL;
    if (batch <= 0 || vocab <= 0 || batch > 65535 || vocab > kMaxVocab || s->row_offset < 0) return KIVI_ERR_SHAPE;
    if (peer_buffers && (!step || !err || world < 1 || rank < 0 || rank >= world || world > 256)) return KIVI_ERR_SHAPE;
    int S = cdiv(vocab, kMinSlice);
    S = S < kMaxCluster ? S : kMaxCluster;
    const int L = cdiv(vocab, S);
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    static std::atomic<unsigned long long> optin{0};
    rc = ensure_dynamic_smem(sample_exchange_kernel, kMaxSlice * (int)sizeof(float), di.ordinal, optin);
    if (rc) return rc;
    Params p;
    p.logits = (const float*)logits; p.V = vocab; p.L = L;
    p.temperature = s->temperature; p.top_k = s->top_k; p.top_p = s->top_p;
    p.seed = (const u64*)s->seed; p.counter = (const long long*)s->counter; p.row_offset = s->row_offset;
    p.next_local = (long long*)next_local; p.ids_feedback = (long long*)ids_feedback;
    p.x = TokenExchange{(long long* const*)peer_buffers, batch, rank, world, (const int*)step, (int*)err};
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(S, batch, 1); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = (size_t)L * sizeof(float);
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = S; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, sample_exchange_kernel, p);
    if (e != cudaSuccess) return (int)e;
    return post_launch();
}
