// kivi_common.cuh -- shared device helpers for libkivi_b200 (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/kivi_b200.h"

#ifndef __CUDA_ARCH__
#define KIVI_HOST_ONLY 1
#endif
#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libkivi_b200 is written for sm_100a (B200) only"
#endif

#include <atomic>

namespace kivi {

extern std::atomic<unsigned long long> g_launch_count;   // host-side counter (kivi_api.cu)

inline int post_launch() {
    g_launch_count.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? KIVI_OK : (int)e;
}

// Properties of the CURRENT device of the calling thread, cached per device ordinal (kivi_api.cu): a process may drive
// several GPUs (device_map="auto" in the reference), and every limit / opt-in below is per device.
constexpr int kMaxDevices = 64;
struct DeviceInfo { int ordinal, num_sms, max_smem_optin; };
int device_info(DeviceInfo* out);            // 0 or a cudaError_t

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) applies to the current device only: `done` is a per-kernel bit mask
// of the device ordinals that already have the opt-in (one static mask per kernel instantiation at the call site).
template <class F>
inline int ensure_dynamic_smem(F kernel, int bytes, int ordinal, std::atomic<unsigned long long>& done) {
    const unsigned long long bit = 1ull << (ordinal & 63);
    if (done.load(std::memory_order_acquire) & bit) return KIVI_OK;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return (int)e;
    done.fetch_or(bit, std::memory_order_release);
    return KIVI_OK;
}

// Tuning knobs from the environment, read ONCE per process (kivi_api.cu); 0 = not set.  Production callers never set
// them (tools/microbench.py, tools/sweep_*.sh do).
struct Tuning { int gqa_g, ctas_per_sm, stages_per_warp, no_pdl, no_mma_gemv; };
const Tuning& tuning();

__host__ __device__ inline int cdiv(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ inline int64_t cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---------------------------------------------------------------------------------------------
// Exact in-register unpack of b-bit codes to fp32 without I2F and without an offset term.
//
// A code field left IN PLACE at bit p of an otherwise zero word (p + bits <= 23) is, read as a
// float, the denormal  c * 2^(p-149)  -- exact, for any c.  FFMA consumes denormal inputs at full
// rate (no .FTZ; this library is never compiled with --use_fast_math), so one LOP3 (AND with an
// immediate mask) per element replaces shift + and + I2F.  The multiplicand carries a 2^90
// pre-scale so that the product is a normal number: with a = x*s (exact in fp32: two fp16
// factors) and a'' = a * 2^90,
//        a'' * as_float(w & (mask << p)) = a * c * 2^(p-59)          (one rounding, in the FMA)
// and the accumulator of element j is rescaled once at the end by the exact power of two
// 2^(59-p_j).  Fields that sit above bit 22 are brought down with ONE shift per word.
//   2-bit: fields 0..10 in place (p = 2i), fields 11..15 from w >> 10 (p = 2i - 10)
//   4-bit: fields 0..4  in place (p = 4i), fields 5..7   from w >> 12 (p = 4i - 12)
// ---------------------------------------------------------------------------------------------
constexpr float kPreScale = 1.2379400392853803e27f;      // 2^90
constexpr float kPreScaleInv = 8.077935669463161e-28f;   // 2^-90

template <int BITS> struct Unpack;

template <> struct Unpack<2> {
    static constexpr int kFpi = 16;
    static constexpr int kSplit = 11;      // first field taken from the shifted word
    static constexpr int kShift = 10;
    __device__ __forceinline__ static int pos(int i) { return i < kSplit ? 2 * i : 2 * i - kShift; }
};
template <> struct Unpack<4> {
    static constexpr int kFpi = 8;
    static constexpr int kSplit = 5;
    static constexpr int kShift = 12;
    __device__ __forceinline__ static int pos(int i) { return i < kSplit ? 4 * i : 4 * i - kShift; }
};

// acc[i] += a2 * denormal(field i of w), i in [0, fpi)
template <int BITS>
__device__ __forceinline__ void fma_word(float (&acc)[32 / BITS], uint32_t w, float a2) {
    using U = Unpack<BITS>;
    const uint32_t hi = w >> U::kShift;
    #pragma unroll
    for (int i = 0; i < U::kFpi; ++i) {
        const uint32_t src = (i < U::kSplit) ? w : hi;
        const uint32_t m = src & (((1u << BITS) - 1u) << U::pos(i));
        acc[i] = fmaf(a2, __uint_as_float(m), acc[i]);
    }
}

// exact rescale factor 2^(59 - p_i) for accumulator i
template <int BITS>
__device__ __forceinline__ float field_rescale(int i) {
    return __uint_as_float((uint32_t)(127 + 59 - Unpack<BITS>::pos(i)) << 23);
}

// fp16( fp32(a / s) ) -- the reference's `data.div_(scale)` on fp16 tensors (quant/new_pack.py:240: ATen divides in fp32 and
// rounds to fp16) -- bit-exact WITHOUT the IEEE division in the common case.  r = RN32(1 / s) (per group, __frcp_rn); q' = a * r
// is within 2 ulp of RN32(a / s), so both round to the same fp16 unless q' lies within a few ulp of an fp16 rounding boundary
// (the 13 dropped mantissa bits == 0x1000); only then -- about one element in a thousand -- or in the fp16 subnormal range, or
// for NaN (0 / 0 of a flat group) the exact division runs.  The division was ~half of the ~35 instructions a quantised element
// costs; every pack path (public pack, prefill, K flush, V token) is bound by that arithmetic, not by HBM.
__device__ __forceinline__ __half quot_to_half(float a, float s, float r) {
    float q = a * r;
    const uint32_t b = __float_as_uint(q);
    const bool sure = ((b & 0x1fffu) - 0x0ffcu > 8u) && (q >= 6.103515625e-05f || q == 0.f);
    if (!sure) q = __fdiv_rn(a, s);
    return __float2half_rn(q);
}

__device__ __forceinline__ float warp_sum(float v) {
    #pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// Token sampling + exchange, shared by the greedy (kivi_model.cu) and the sampling (kivi_sample.cu) kernels.
// ---------------------------------------------------------------------------------------------
// The argmax order of torch.argmax: a NaN beats every number, and among NaNs, as among equal maxima, the lower index wins.
// It is a total order, so every reduction tree over (value, index) pairs ends at the same pair.
__device__ __forceinline__ bool argmax_takes(float best, int bi, float ov, int oi) {
    return (ov != ov) ? (!(best != best) || oi < bi) : (!(best != best) && (ov > best || (ov == best && oi < bi)));
}

__device__ __forceinline__ void warp_argmax(float& best, int& bi) {
    #pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (argmax_takes(best, bi, ov, oi)) { best = ov; bi = oi; }
    }
}

// The ids of one step travel to every data-parallel replica (kivi_greedy_sample_exchange_f32 in include/kivi_b200.h):
//   peer[p]  : rank p's buffer: int64 tokens[2][world * B] (double-buffered by step parity), then uint64 arrived[world]
//   step     : device counter, incremented by the caller BEFORE the launch (inside the same CUDA graph)
// peer == nullptr: one GPU, no exchange.
struct TokenExchange {
    long long* const* peer;
    int B, rank, world;
    const int* step;
    int* err;
};

// One thread per sequence: the id of sequence b goes to next_local, ids_feedback (may be NULL) and -- replicas -- into this
// rank's slot of EVERY rank's token buffer with plain peer stores over NVLink / NVSwitch, then releases a per-rank arrival
// counter on every peer.
__device__ __forceinline__ void exchange_publish(long long tok, int b, long long* next_local, long long* ids_feedback,
                                                 const TokenExchange& x) {
    next_local[b] = tok;
    if (ids_feedback) ids_feedback[b] = tok;
    if (x.peer) {
        const int step = *x.step;
        const long long slot = (long long)(step & 1) * x.world * x.B + (long long)x.rank * x.B + b;
        for (int p = 0; p < x.world; ++p) x.peer[p][slot] = tok;
        __threadfence_system();                                             // the ids are visible system-wide before the arrivals
        for (int p = 0; p < x.world; ++p)
            atomicAdd_system(reinterpret_cast<unsigned long long*>(x.peer[p] + 2ll * x.world * x.B + x.rank), 1ull);
    }
}

// Threads tid < world of ONE block wait (bounded) until all ranks' ids of this step have arrived in this rank's buffer; on
// time-out *err = 1 instead of hanging the GPU.
__device__ __forceinline__ void exchange_wait(const TokenExchange& x, int tid) {
    if (!x.peer || tid >= x.world) return;
    const unsigned long long want = (unsigned long long)(*x.step) * (unsigned long long)x.B;
    const volatile unsigned long long* cnt =
        reinterpret_cast<const volatile unsigned long long*>(x.peer[x.rank] + 2ll * x.world * x.B + tid);
    long long spins = 0;
    while (*cnt < want) {
        if (++spins > (1ll << 24)) { *x.err = 1; break; }                  // ~ a second: a peer is gone
        __nanosleep(64);
    }
    __threadfence_system();
}

}  // namespace kivi
