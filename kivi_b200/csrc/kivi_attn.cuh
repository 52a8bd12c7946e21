// kivi_attn.cuh -- KIVI decode attention over the blocked cache (sm_100a): two barrier-free launches.
//
// Replaces the ~30 launches of the reference's decode branch (models/llama_kivi.py:314-399): q.Kq^T with
// in-register dequantisation, the fp16 K window, scale, mask, fp32 softmax, p.Vq, the fp16 V window, the
// fp16 add, and the per-unit cache data movement (window append, K flush, V token pack).  Rounding points
// of the reference are reproduced (fp16 logits -> fp16 scale -> fp32 softmax -> fp16 probs -> fp16 partial
// outputs -> fp16 add).
//
// Execution model: EVERY WARP IS AN AUTONOMOUS WORKER -- no CTA barrier anywhere, no per-unit tail.
//   qk_kernel   the (unit, pseudo-block) sequence [K blocks | fp16 K window items | new token] of all units is cut
//               into one contiguous range per warp.  A warp writes the scaled fp16 logits of its pseudo-blocks to the
//               workspace row and ONE (max, sum exp) statistics pair per unit it touches (online softmax per lane).
//   sv_kernel   the (unit, pseudo-block) sequence [V blocks | fp16 V window items | new token] of all units is cut
//               into one contiguous range per warp.  A warp combines the row's statistics into (M, S) -- the same
//               instructions on the same data in every warp, hence bit-identical -- turns the logits slice of its
//               block into fp16 probabilities in place in shared memory (they arrive with the block through the
//               same bulk-copy group), accumulates across the blocks of a unit, and writes one partial record per
//               unit.  The LAST warp to arrive for a unit (atomic counter) adds the records in a fixed order,
//               rounds, writes the output and performs the unit's cache update.
//   Data movement: each warp owns S private shared-memory stages and streams its own items HBM -> smem with
//   1-D bulk copies (cp.async.bulk = the TMA engine, SASS UBLKCP, L2 evict-first) completing on the stage's
//   mbarrier; right after consuming a stage its elected lane issues the copy of the item S positions ahead
//   (fence.proxy.async orders its reads before the async write).
//
// Arithmetic of a packed block (128 inner x 128 outer, kivi_decode.cuh):
//     sum_i x_i * (s_i,G * c_i,o + z_i,G) = sum_i (x_i * s_i,G) * c_i,o  +  sum_i x_i * z_i,G
//   SIMT needs one LOP3 + one FFMA per code and is bound by the 16-lane ALU pipe (measured: 2.5 TB/s
//   equivalent, profiles/r01_decode_attention_ncu_summary.txt).  Here the tensor cores are an UNPACK
//   AMORTISER: the only per-code work left is isolating the field, ONE LOP3 per PAIR of codes:
//     A (16 outer x 16 inner, fp16)  codes as fp16 denormals code * 2^(P-24), P >= 4 (exact in mma.sync: Lay<>::shr)
//     B (16 inner x 8 cols,  fp16)  column (group, head, part): x_i * s_i,G split EXACTLY with two half2
//                                   instructions: hi = x*s (rounded), lo = fma(x, s, -hi) (the residual of
//                                   an fp16 product is an fp16); G query heads share the MMA (GQA is free)
//     C (16 outer x 8 cols,  fp32)  row o, columns (G(o), h, hi | lo) are the wanted sums; the other
//                                   columns are cross terms and are ignored.  Products exact, fp32 accumulate.
//   The zero term is one more MMA per 16 inner indices with exact fp16 operands (rows = z_G, cols = x_h).
#pragma once
#include <cstdlib>
#include "kivi_decode.cuh"

// tuning knobs of the chunk loop (tools/build_variants.py measures the alternatives)
#ifndef KIVI_UNROLL
#define KIVI_UNROLL 8
#endif
constexpr int kChunkUnroll = KIVI_UNROLL;
#ifndef KIVI_Z_SIMT
#define KIVI_Z_SIMT 0                    // 1: zero term of G == 1 kernels with FFMAs instead of one MMA per chunk (measured: see DESIGN.md)
#endif
#ifndef KIVI_EVICT_FIRST
#define KIVI_EVICT_FIRST 1
#endif
#ifndef KIVI_SHIFT_IMAD
#define KIVI_SHIFT_IMAD 0
#endif
#ifndef KIVI_PRED_FINALIZE
#define KIVI_PRED_FINALIZE 1             // 0: the round-1 epilogue (selects); A/B builds
#endif
// 1: the p.V kernel does not wait for the whole q.K^T grid (griddepcontrol.wait) but, unit by unit, for the q.K^T ranges of
// that unit (release / acquire counters in the workspace): a p.V CTA starts working the moment ITS SM's q.K^T CTA has left,
// while slower SMs are still in their q.K^T tail.  Correct (tests pass in both modes) but MEASURED SLOWER: the release fence
// of every (warp, unit) visit of q.K^T and the acquire round trip of every p.V visit cost more than the hand-over they
// save (cfg 2: 0.0992 vs 0.0953 ms per call, cfg 3 0.137 vs 0.131, B = 128 0.346 vs 0.334; gpurun_out/r2m, DESIGN.md 6).
#ifndef KIVI_EARLY_COMMIT
#define KIVI_EARLY_COMMIT 1              // 1: the units' cache updates run at the START of the p.V kernel (spread over its warps); 0: in the last arriver
#endif
#ifndef KIVI_UNIT_FLAGS
#define KIVI_UNIT_FLAGS 0
#endif
// 1: the units' cache updates (V-token pack, window appends) are done by the q.K^T warps AFTER their ranges, one unit per
// ticket of a device counter (a finished warp draws until none is left), instead of at the start of the p.V kernel, where they
// sit on the critical path of 43 % of its warps (1024 units over 2368 warps: 96 % of the latest tenth of the p.V warps are
// committing warps, +2.9 us each; profiles/r02_timeline_commit.txt).  Correct (GPU suite + memcheck pass) but MEASURED SLOWER:
// too few q.K^T warps finish early enough, the draws run until 47.9 us instead of the grid ending at 45.6 us, and the p.V
// kernel gains only 1.3 us of it back (cfg 2: 0.0955 vs 0.0923 ms per call, cfg 3 0.1312 vs 0.1283, B = 128 0.3296 vs 0.3249).
#ifndef KIVI_COMMIT_IN_QK
#define KIVI_COMMIT_IN_QK 0
#endif
#if KIVI_COMMIT_IN_QK && KIVI_UNIT_FLAGS
#error "KIVI_COMMIT_IN_QK relies on the grid dependency between the two kernels (the ticket reset); KIVI_UNIT_FLAGS removes it"
#endif
#ifndef KIVI_PREFETCH_SV
#define KIVI_PREFETCH_SV 0               // n > 0: a finished q.K^T warp requests the first n packed V items of "its" p.V range into L2
#endif
// Latency fixes read off the ncu source counters of the cfg-2 call (profiles/r02_latency_fixes.txt); A/B per shape, graph-timed:
//   KIVI_Q_FIRST         q.K^T issues ONE stage, fetches q, then the other stages (0: all stages first).  G = 1: -1.0 % per call
//                        (cfg 2); G = 4: 0 ... +0.7 % (cfg 3 / cfg 4) -> applied to the G = 1 kernels only.
//   KIVI_WIN_LOGITS_BULK the logits of a V window item travel with its bulk-copy group instead of a dependent global load.
//                        G = 1: -0.4 % (cfg 2); G = 4 (4 extra copies per item): +0.3 ... +0.5 % -> G = 1 only.
//   KIVI_REL_ARRIVE      the p.V arrival as a release, the acquire only in the last arriver: +0.4 % (cfg 2) / -0.4 % (cfg 3),
//                        i.e. nothing: off.
// 1: the inputs of a warp's cache update travel as the first item of its stage queue (see the p.V kernel).  The first stages
// are then issued by all warps within 0.5 us of each other (p90 of "first stage issued": 47.6 instead of 54 us), but the call
// gets SLOWER (cfg 2 0.0939 vs 0.0924 ms, B = 128 0.3264 vs 0.3218, same box): the committing warps start with one packed block
// in flight instead of two.  Off.
#ifndef KIVI_COMMIT_ASYNC
#define KIVI_COMMIT_ASYNC 0
#endif
// 1: a p.V arrival that is followed by another visit of the warp is issued after that visit's first item, when the record
// stores have landed and the release fence returns at once (the fence + atomic + L1 invalidation of an arrival are 7.4 % of the
// kernel's warp time).  Only 29 % of the arrivals have a visit behind them; MEASURED SLOWER: cfg 2 0.0894 vs 0.0887 ms, B = 128
// 0.3177 vs 0.3153 (the test in the item loop costs more than the hidden fences save).  Off.
#ifndef KIVI_DEFER_ARRIVE
#define KIVI_DEFER_ARRIVE 0
#endif
#ifndef KIVI_Q_FIRST
#define KIVI_Q_FIRST 1
#endif
#ifndef KIVI_REL_ARRIVE
#define KIVI_REL_ARRIVE 0
#endif
#ifndef KIVI_WIN_LOGITS_BULK
#define KIVI_WIN_LOGITS_BULK 1
#endif
// The kernel parameters are __grid_constant__: the noinline cache-update callees (commit_unit, k_flush_slice) take `const
// AttnParams&`, and without the qualifier every thread of the p.V kernel first copied the 350-byte struct to local memory --
// 26 MB of local stores at the very moment the grid starts (ncu: STL.128 rows with lg_throttle stalls, 3 % of the kernel's warp
// time; stack frame 352 -> 112 bytes).  -3.0 % per cfg-2 call (0.0923 -> 0.0896 ms).  -DKIVI_GRID_CONSTANT=0 for the A/B.
#ifndef KIVI_GRID_CONSTANT
#define KIVI_GRID_CONSTANT 1
#endif
#if KIVI_GRID_CONSTANT
#define KIVI_PARAM_QUAL __grid_constant__
#else
#define KIVI_PARAM_QUAL
#endif
template <int G> struct Lat { static constexpr bool q_first = KIVI_Q_FIRST && G == 1, win_bulk = KIVI_WIN_LOGITS_BULK && G == 1; };
#ifndef KIVI_COMMIT_LATE
#define KIVI_COMMIT_LATE 0               // 1: the early cache updates run after the warp's first stages are in flight instead of before the grid-dependency wait
#endif

namespace kivi {

int make_desc(const kivi_cache_t* k, CacheDesc* d);

// Warps per CTA (they never synchronise with each other).  16 = ONE CTA per SM: with two CTAs of 8 warps the SM's warp
// scheduler favours the older CTA, whose warps finish ~25 % earlier and leave the SM half empty for the last ~10 us of a
// 50 us kernel (tools/timeline.py, profiles/r01_timeline_static_ranges.txt); sixteen warps of one age finish together.
#ifndef KIVI_CW
#define KIVI_CW 16
#endif
constexpr int kCW = KIVI_CW;
#ifndef KIVI_MINB
#define KIVI_MINB (KIVI_CW >= 16 ? 1 : 2)   // CTAs per SM the kernels are compiled for (register budget) and launched with
#endif
// The 4-bit K kernels that serve four query heads per KV head run 12 warps per CTA: at 16 warps their accumulators and the
// four heads' B fragments spill (128 registers), at 12 they have 170 and the 4-bit block loop needs fewer warps to cover its
// latencies (half the unpack instructions per byte).  Measured, one B200, per call (profiles/r02_warps_per_cta.txt):
// cfg 4 (K4V4 g64, G = 4) 0.1325 vs 0.1410 ms, K4V4 g128 G = 4 0.0798 vs 0.0857 ms; G = 1 equal, G = 2 -1 %; 14 / 11 / 10
// warps slower; the 2-bit kernels lose 5 - 11 % at 12 warps (cfg 2, cfg 3) and stay at 16.
#ifndef KIVI_CW_K4G4
#define KIVI_CW_K4G4 12
#endif
template <int KB, int G> struct WarpsPerCta { static constexpr int k = (KB == 4 && G == 4 && KIVI_CW >= 16) ? KIVI_CW_K4G4 : kCW; };
// A pipeline stage holds kHalfChunks of the 8 chunks (16 inner indices each) of a packed block: 8 = whole blocks
// (one 6 KB bulk copy), 4 = half blocks.  Measured (tools/sweep_occupancy.sh, profiles/): half blocks allow 3 CTAs
// per SM (24 warps) but cost +25 % instructions and more, smaller copies -> 175 us vs 140 us per cfg-2 layer.
constexpr int kHalfChunks = 8;
constexpr int kParts = 8 / kHalfChunks;     // stage-items per packed block
constexpr int kPartTokens = 16 * kHalfChunks;   // inner indices (V: tokens) per stage-item
constexpr int kResTile = 16;                // tokens per fp16-window item (256 B each): one MMA tile of tokens
constexpr int kResBytes = kResTile * kD * 2;
constexpr float kRcpSqrtD = 1.0f / 11.313708f;   // ATen: x * (1.0f / float(math.sqrt(128)))  (llama_kivi.py:339)
// probabilities are kept x 2^6 while they feed the MMAs: exact, and it keeps the fp16 residual fma(p, s, -hi) of
// small probabilities out of the denormal range
constexpr float kProbScale = 64.f, kProbScaleInv = 1.f / 64.f;

// Programmatic dependent launch (PDL): a kernel launched with the programmatic-serialization attribute may start while its
// predecessor in the stream is still draining; pdl_wait() blocks until the predecessor has completed and flushed, and
// pdl_trigger() tells the runtime that the successor may start launching.  Both are no-ops for ordinary launches.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;"); }

#if KIVI_TIMELINE
// per-warp timestamps (globaltimer ns) of the two kernels: [kernel][warp][entry, first data, blocks done, exit, smid]
static __device__ unsigned long long g_timeline[2][4096][8];   // one copy per translation unit
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define KIVI_TL(k, w, i) do { if (lane == 0 && (w) < 4096) { g_timeline[k][w][i] = gtime(); if ((i) == 0) { unsigned sm_; asm volatile("mov.u32 %0, %%smid;" : "=r"(sm_)); g_timeline[k][w][4] = sm_; } } } while (0)
// every translation unit has its own copy (no relocatable device code), and a kernel instantiated in two of them (the
// q.K^T kernel does not depend on v_bits) writes whichever copy the linker kept: kivi_debug_timeline merges all of them
static inline int timeline_fetch(unsigned long long* host_out) {
    return (int)cudaMemcpyFromSymbol(host_out, g_timeline, sizeof(unsigned long long) * 2 * 4096 * 8);
}
#else
#define KIVI_TL(k, w, i) do {} while (0)
#endif

struct Workspace {                     // carved from the caller's buffer (kivi_decode_workspace_bytes)
    __half* lg; long long ld;          // [B*H][ld] scaled logits (fp16), ld % 128 == 0
    float2* stats; int stat_cap;       // [B*H][stat_cap] (max, sum exp(x - max)) per qk item
    float* part; int part_cap;         // [n_units][part_cap][G][2][128] partial outputs (packed | window)
    int* count;                        // [n_units] arrivals of sv ranges; the last arriver resets it to 0
    int* ready;                        // [n_units] q.K^T ranges of the unit that have published logits + statistics (reset by the finaliser)
    int* ticket;                       // [1] next unit whose cache update is up for grabs (q.K^T warps draw, the p.V kernel resets it to 0)
};

struct AttnParams {
    CacheDesc c;
    const __half* q; const __half* k_new; const __half* v_new; const __half* mask;
    __half* out; __half* dbg_logits; __half* dbg_probs;
    long long dbg_stride;
    Workspace w;
    int stage_bytes, spw /*stages per warp*/, hchunks, n_units, nw_eff /*warps that own an sv range*/;
    int max_kv_len;                     // what the workspace rows were sized for
    const int* seq_start;               // NULL, or [B]: positions < seq_start[b] of sequence b are left padding (qk_kernel<PAD>)
};

struct Sched {                          // per-step constants, identical for every unit
    int tk, r, tv, L, vhead, T, seg1;
    int n_kb, n_kr, n_vb, vr1, n_vr;
    int ipu;                            // qk items per unit: K blocks, K window items, the new token
    int bpu;                            // sv pseudo-blocks per unit: V blocks, V window items, the new token
};

__device__ __forceinline__ Sched make_sched(const CacheDesc& c) {
    Sched s;
    s.tk = c.state[ST_TK]; s.r = c.state[ST_R]; s.tv = c.state[ST_TV]; s.L = c.state[ST_L]; s.vhead = c.state[ST_VHEAD];
    s.T = s.tk + s.r + 1;
    s.n_kb = cdiv(s.tk, kBlockTokens);
    s.n_kr = cdiv(s.r, kResTile);
    s.n_vb = cdiv(s.tv, kBlockTokens);
    s.seg1 = min(s.L, c.v_res_cap - s.vhead);
    s.vr1 = cdiv(s.seg1, kResTile);
    s.n_vr = s.vr1 + cdiv(s.L - s.seg1, kResTile);
    s.ipu = s.n_kb + s.n_kr + 1;
    s.bpu = s.n_vb + s.n_vr + 1;
    return s;
}

// The device-side lengths are trusted by every address computation below; a C-ABI caller that stepped past the sizes it
// declared (max_kv_len, window capacities) must not corrupt memory: the kernels return without touching anything and
// leave KIVI_STATE_ERR_CAPACITY in state[6] (surfaced by kivi_cache_read_state).
__device__ __forceinline__ bool sched_ok(const Sched& s, const CacheDesc& c, int max_kv_len) {
    return s.tk >= 0 && s.tv >= 0 && s.r >= 0 && s.L >= 0 && s.r < c.R && s.L <= c.R && s.T <= max_kv_len &&
           s.tv + 1 <= max_kv_len && s.vhead >= 0 && s.vhead < c.v_res_cap && s.tk % c.R == 0;
}

struct Pipe {                           // a warp's private stages
    uint8_t* base; uint64_t* full; int spw, stage_bytes;
    int c_stage, c_par;                 // consumer: current stage and its mbarrier parity
    int i_stage;                        // producer: stage of the next copy
    __device__ __forceinline__ void init(uint8_t* b, uint64_t* f, int spw_, int sb) {
        base = b; full = f; spw = spw_; stage_bytes = sb; c_stage = 0; c_par = 0; i_stage = 0;
    }
    __device__ __forceinline__ uint8_t* cons() const { return base + (size_t)c_stage * stage_bytes; }
    __device__ __forceinline__ void wait() const { mbar_wait(&full[c_stage], (uint32_t)c_par); }
    __device__ __forceinline__ void pop() { if (++c_stage == spw) { c_stage = 0; c_par ^= 1; } }
    __device__ __forceinline__ uint8_t* prod() const { return base + (size_t)i_stage * stage_bytes; }
    __device__ __forceinline__ uint64_t* prod_bar() const { return &full[i_stage]; }
    __device__ __forceinline__ void push() { if (++i_stage == spw) i_stage = 0; }
};

// logits (fp16 kernel output) -> fp16 scaled, the value that enters the softmax
__device__ __forceinline__ __half scale_logit(float acc) {
    return __float2half_rn(__half2float(__float2half_rn(acc)) * kRcpSqrtD);
}

// exp(x) = ex2.approx(x * log2 e), results below 2^-126 flushed to zero: two instructions (__expf adds a range fix-up)
__device__ __forceinline__ float fast_exp(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x * 1.4426950408889634f));
    return y;
}

__device__ __forceinline__ uint32_t h2_as_u32(const __half2 h) { return *reinterpret_cast<const uint32_t*>(&h); }
__device__ __forceinline__ __half2 u32_as_h2(const uint32_t u) { return *reinterpret_cast<const __half2*>(&u); }

// One B-fragment register: column part 0 -> hi = fp16(x*s); part 1 -> lo = x*s - hi (exact: the residual of an fp16
// product is an fp16).
#ifndef KIVI_BPREP2
#define KIVI_BPREP2 1                    // 1: hi, then a PREDICATED fma(x, s, -hi) in the lo lanes (2 instructions); 0: branch-free 3
#endif
__device__ __forceinline__ uint32_t b_prep(uint32_t x2, uint32_t s2, __half2 msel) {
    const __half2 x = u32_as_h2(x2), s = u32_as_h2(s2);
#if KIVI_BPREP2
    __half2 b = __hmul2(x, s);
    if (h2_as_u32(msel) != 0u) b = __hfma2(x, s, __hneg2(b));   // lane-invariant predicate, negation folds into the HFMA2 operand
    return h2_as_u32(b);
#else
    const __half2 nh = __hmul2(__hmul2(x, s), msel);         // nh = hi * (part ? -1 : 0);  b = fma(x, s, nh)
    return h2_as_u32(__hfma2(x, s, nh));
#endif
}

// exact power of two 2^(24 - P) that undoes the denormal scaling of the fields of MMA mm
template <int BITS>
__device__ __forceinline__ float inv_pos_scale(int mm) {
    return __uint_as_float((uint32_t)(127 + 24 - Lay<BITS>::bitpos(mm % Lay<BITS>::F)) << 23);
}

// column bookkeeping of the B fragments (G query heads, NG outer groups per block)
template <int G, int GS>
struct Cols {
    static constexpr int NG = 128 / GS;               // outer groups per block (g >= 32 -> NG <= 4)
    static constexpr int GPF = 4 / G;                  // groups per B fragment (8 columns = GPF x G heads x hi/lo)
    static constexpr int NF = (NG + GPF - 1) / GPF;    // B fragments per 16 inner indices
};

// ------------------------------------------------------------------------------------------------
// Half a packed block (inner indices 16*c0 .. 16*c0+63, 128 outer) on the tensor cores.
//   st      : the half block in shared memory: 4 chunks of codes, then the 4 chunks of meta
//   getx    : (chunk c, head h, &xa, &xb) -> the lane's x values (half2) of inner indices 16c+2t+{0,1} and
//             16c+2t+{8,9} for head h (c = chunk within the whole block)
//   acc[mm] : accumulators of MMA mm (outer rows 16mm .. 16mm+15): lane (g8, t) holds rows g8 / g8+8 of
//             columns 2t, 2t+1 = (group-in-fragment t / G, head t % G, hi | lo)
//   zc      : zero-term accumulator: row g8 = group min(g8 >> 1, NG-1), columns 2t, 2t+1 = head t % G
// ------------------------------------------------------------------------------------------------
template <int BITS, int G, int GS, bool INIT, class XF>
__device__ __forceinline__ void mma_half(const uint8_t* st, int c0, XF&& getx, float (&acc)[8][4], float (&zc)[4], int lane)
{
    using L = Lay<BITS>;
    using CL = Cols<G, GS>;
    constexpr int NG = CL::NG, GPF = CL::GPF, NF = CL::NF;
    const int g8 = lane >> 2, t = lane & 3;
    const int hb = (g8 % (2 * G)) >> 1;                 // head of this lane's B column
    const int gi = g8 / (2 * G);                        // group-in-fragment of this lane's B column
    const int gz = min(g8 >> 1, NG - 1);                // group of this lane's A rows in the zero-term MMA
    const __half2 msel = (g8 & 1) ? __float2half2_rn(-1.f) : __float2half2_rn(0.f);
    const uint8_t* meta = st + kHalfChunks * L::kChunkBytes + t * 16;
    constexpr uint32_t kField = ((1u << BITS) - 1u) * 0x00010001u;
    #pragma unroll (kChunkUnroll)
    for (int cl = 0; cl < kHalfChunks; ++cl) {
        uint32_t xa, xb;
        getx(c0 + cl, hb, xa, xb);
        // {z(2t,2t+1), s(2t,2t+1), z(2t+8,2t+9), s(2t+8,2t+9)} of group gz: as is, the A operand of the zero-term MMA
        const uint4 mz = *reinterpret_cast<const uint4*>(meta + (cl * NG + gz) * 64);
        if (KIVI_Z_SIMT && G == 1) {
            // zero term on the FMA pipe: this lane's four inner indices of (group gz); zc[0] collects the lane's partial sum
            const float2 x0 = __half22float2(u32_as_h2(xa)), x1 = __half22float2(u32_as_h2(xb));
            const float2 z0 = __half22float2(u32_as_h2(mz.x)), z1 = __half22float2(u32_as_h2(mz.z));
            float zp = (INIT && cl == 0) ? x0.x * z0.x : fmaf(x0.x, z0.x, zc[0]);
            zp = fmaf(x0.y, z0.y, zp); zp = fmaf(x1.x, z1.x, zp); zc[0] = fmaf(x1.y, z1.y, zp);
        } else if (INIT && cl == 0) mma_16816_init(zc, mz.x, mz.y, mz.z, mz.w, xa, xb);   // first chunk of a block: D = A * B
        else mma_16816(zc, mz.x, mz.y, mz.z, mz.w, xa, xb);
        uint32_t b0[NF], b1[NF];
        if (G == 1 && NF == 1) {                        // the B column's group is gz
            b0[0] = b_prep(xa, mz.y, msel); b1[0] = b_prep(xb, mz.w, msel);
        } else {
            #pragma unroll
            for (int f = 0; f < NF; ++f) {
                const int grp = min(f * GPF + gi, NG - 1);
                const uint4 ms = *reinterpret_cast<const uint4*>(meta + (cl * NG + grp) * 64);
                b0[f] = b_prep(xa, ms.y, msel); b1[f] = b_prep(xb, ms.w, msel);
            }
        }
        #pragma unroll
        for (int sl = 0; sl < L::kSlabs; ++sl) {
            const uint4 w4 = *reinterpret_cast<const uint4*>(st + (cl * L::kSlabs + sl) * 512 + lane * 16);
            const uint32_t w[4] = {w4.x, w4.y, w4.z, w4.w};
            uint32_t wl4[4], wr4[4], wr6[4], wr8[4];    // the shifted copies a bit width needs (the others fold away)
            #pragma unroll
            for (int r = 0; r < 4; ++r) {                 // right shifts as IMAD.HI: the FMA pipe has room, the ALU pipe (LOP3) does not
#if KIVI_SHIFT_IMAD
                wl4[r] = w[r] << 4; wr4[r] = __umulhi(w[r], 1u << 28); wr6[r] = __umulhi(w[r], 1u << 26); wr8[r] = __umulhi(w[r], 1u << 24);
#else
                wl4[r] = w[r] << 4; wr4[r] = w[r] >> 4; wr6[r] = w[r] >> 6; wr8[r] = w[r] >> 8;
#endif
            }
            #pragma unroll
            for (int j = 0; j < L::F; ++j) {
                uint32_t a[4];
                #pragma unroll
                for (int r = 0; r < 4; ++r) {
                    const int sh = L::shr(j);
                    const uint32_t src = sh == -4 ? wl4[r] : sh == 0 ? w[r] : sh == 4 ? wr4[r] : sh == 6 ? wr6[r] : wr8[r];
                    a[r] = src & (kField << L::bitpos(j));
                }
                const int mm = sl * L::F + j;
                const int f = ((16 * mm) / GS) / GPF;
                if (INIT && cl == 0) mma_16816_init(acc[mm], a[0], a[1], a[2], a[3], b0[f], b1[f]);
                else mma_16816(acc[mm], a[0], a[1], a[2], a[3], b0[f], b1[f]);
            }
        }
    }
}

// The lane's zero term for every outer group: Z[head t % G][grp] lives in the lanes with g8 = 2 * grp.
template <int G, int GS>
__device__ __forceinline__ void gather_z(const float (&zc)[4], int lane, float (&zsel)[Cols<G, GS>::NG]) {
    float z = zc[0];
    if (KIVI_Z_SIMT && G == 1) {                        // the four t-lanes of a g8 row hold partial sums of its group
        z += __shfl_xor_sync(0xffffffffu, z, 1);
        z += __shfl_xor_sync(0xffffffffu, z, 2);
    }
#if KIVI_PRED_FINALIZE
    if (G == 1 && GS == 32) {                           // finalize() reads zsel[t] only (t = lane & 3): one shuffle, source lane 8t + t
        const float zt = __shfl_sync(0xffffffffu, z, 9 * (lane & 3));
        #pragma unroll
        for (int grp = 0; grp < Cols<G, GS>::NG; ++grp) zsel[grp] = zt;
        return;
    }
#endif
    #pragma unroll
    for (int grp = 0; grp < Cols<G, GS>::NG; ++grp)
        zsel[grp] = __shfl_sync(0xffffffffu, z, 8 * grp + (lane & 3));
}

// branch-free v[t] for t = (t2, t1): three SELP (the compiler turns long ?: chains over registers into branches)
__device__ __forceinline__ float selp(float a, float b, bool p) {
    float r;
    asm("{ .reg .pred q; setp.ne.b32 q, %3, 0; selp.f32 %0, %2, %1, q; }" : "=f"(r) : "f"(a), "f"(b), "r"((int)p));
    return r;
}
__device__ __forceinline__ float sel4(float v0, float v1, float v2, float v3, bool t1, bool t2) {
    return selp(selp(v0, v1, t1), selp(v2, v3, t1), t2);
}

// Hand every (slot, outer row, value) this lane owns to `emit`: value = ((hi + lo) * 2^(24-P) + Z) * post for its
// head t % G; `slot` is a compile-time index (< kSlots) of the value within the lane.  Lane (g8, t) owns rows
// g8 / g8+8 of the MMAs whose group-in-fragment is t / G.
template <int G, int GS> struct Slots { static constexpr int k = (G == 1 && GS == 32) ? 4 : 16; };

template <int BITS, int G, int GS, class EF>
__device__ __forceinline__ void finalize(const float (&acc)[8][4], const float (&zsel)[Cols<G, GS>::NG], int lane,
                                         float post, EF&& emit)
{
    constexpr int GPF = Cols<G, GS>::GPF;
    const int g8 = lane >> 2, t = lane & 3;
    if (G == 1 && GS == 32) {
        // lane t owns MMAs 2t and 2t+1 (group t).
#if KIVI_PRED_FINALIZE
        // Four PREDICATED copies of the eight FADD / FFMA (one per value of t, compile-time accumulator indices and scales):
        // they run on the FMA pipe, which idles, instead of 33 selects on the ALU pipe, which is the one that binds.
        float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
        #pragma unroll
        for (int v = 0; v < 4; ++v) {
            if (t == v) {
                const float sl = inv_pos_scale<BITS>(2 * v) * post, sh = inv_pos_scale<BITS>(2 * v + 1) * post, zt = zsel[v] * post;
                v0 = fmaf(acc[2 * v][0] + acc[2 * v][1], sl, zt);
                v1 = fmaf(acc[2 * v][2] + acc[2 * v][3], sl, zt);
                v2 = fmaf(acc[2 * v + 1][0] + acc[2 * v + 1][1], sh, zt);
                v3 = fmaf(acc[2 * v + 1][2] + acc[2 * v + 1][3], sh, zt);
            }
        }
        const int o = 32 * t + g8;
        emit(0, o, v0);
        emit(1, o + 8, v1);
        emit(2, o + 16, v2);
        emit(3, o + 24, v3);
#else
        // pick them with selects instead of 8 predicated copies of the tail
        const bool t1 = t & 1, t2 = t & 2;
        float lo[4], hi[4];
        #pragma unroll
        for (int e = 0; e < 4; ++e) {
            lo[e] = sel4(acc[0][e], acc[2][e], acc[4][e], acc[6][e], t1, t2);
            hi[e] = sel4(acc[1][e], acc[3][e], acc[5][e], acc[7][e], t1, t2);
        }
        const float sl = sel4(inv_pos_scale<BITS>(0), inv_pos_scale<BITS>(2), inv_pos_scale<BITS>(4), inv_pos_scale<BITS>(6), t1, t2) * post;
        const float sh = sel4(inv_pos_scale<BITS>(1), inv_pos_scale<BITS>(3), inv_pos_scale<BITS>(5), inv_pos_scale<BITS>(7), t1, t2) * post;
        const float zt = sel4(zsel[0], zsel[1], zsel[2], zsel[3], t1, t2) * post;
        const int o = 32 * t + g8;
        emit(0, o, fmaf(lo[0] + lo[1], sl, zt));
        emit(1, o + 8, fmaf(lo[2] + lo[3], sl, zt));
        emit(2, o + 16, fmaf(hi[0] + hi[1], sh, zt));
        emit(3, o + 24, fmaf(hi[2] + hi[3], sh, zt));
#endif
    } else {
        const int gi_l = t / G;
        #pragma unroll
        for (int mm = 0; mm < 8; ++mm) {
            const int grp = (16 * mm) / GS;
            if (grp % GPF == gi_l) {
                const float sc = inv_pos_scale<BITS>(mm) * post, zt = zsel[grp] * post;
                emit(2 * mm, 16 * mm + g8, fmaf(acc[mm][0] + acc[mm][1], sc, zt));
                emit(2 * mm + 1, 16 * mm + g8 + 8, fmaf(acc[mm][2] + acc[mm][3], sc, zt));
            }
        }
    }
}

// the same ownership walk over per-lane slot values (the running sums of the p.V kernel)
template <int G, int GS, class EF>
__device__ __forceinline__ void walk_slots(const float (&run)[Slots<G, GS>::k], int lane, EF&& emit)
{
    constexpr int GPF = Cols<G, GS>::GPF;
    const int g8 = lane >> 2, t = lane & 3;
    if (G == 1 && GS == 32) {
        #pragma unroll
        for (int e = 0; e < 4; ++e) emit(32 * t + g8 + 8 * e, run[e]);
    } else {
        const int gi_l = t / G;
        #pragma unroll
        for (int mm = 0; mm < 8; ++mm) {
            if (((16 * mm) / GS) % GPF == gi_l) {
                emit(16 * mm + g8, run[2 * mm]);
                emit(16 * mm + g8 + 8, run[2 * mm + 1]);
            }
        }
    }
}

// quantise one value with its group's (min, scale): quant/new_pack.py:238-241 (rint follows)
__device__ __forceinline__ float q_code(float x, float mnf, float scf, float rcp, float maxq) {
    const __half t1 = __float2half_rn(x - mnf);
    const __half t2 = quot_to_half(__half2float(t1), scf, rcp);
    return fminf(fmaxf(__half2float(t2), 0.f), maxq);
}

// ------------------------------------------------------------------------------------------------
// cache data movement of one unit (models/llama_kivi.py:343-356, :386-399), executed by ONE warp (the last
// arriver of the unit); cold path, kept out of line.  scratch: 128 bytes of shared memory private to the warp.
// ------------------------------------------------------------------------------------------------
// the inputs of a unit's cache update: fetched before the warp's arrival for the unit, so that their round trip overlaps the
// arrival's (under load a dependent global round trip costs ~2 us and the finalisation sits at the very end of a warp's range)
struct CommitIn { uint4 vnew4, knew4; uint2 vold; };

__device__ __forceinline__ CommitIn commit_fetch(const AttnParams& p, const Sched& s, int u, int lane)
{
    const CacheDesc& c = p.c;
    CommitIn in;
    in.vnew4 = make_uint4(0u, 0u, 0u, 0u); in.knew4 = in.vnew4; in.vold = make_uint2(0u, 0u);
    if (lane < kD / 8) in.vnew4 = __ldg(reinterpret_cast<const uint4*>(p.v_new + (int64_t)u * kD) + lane);
    if (lane >= 16) in.knew4 = __ldg(reinterpret_cast<const uint4*>(p.k_new + (int64_t)u * kD) + (lane - 16));
    if (s.L + 1 > c.R) in.vold = __ldcg(reinterpret_cast<const uint2*>(c.v_res + (int64_t)u * c.v_res_cap * kD + win_off(s.vhead, lane * 4)));
    return in;
}

template <int KB, int VB>
__device__ __noinline__ void commit_unit(const AttnParams& p, const Sched& s, int u, int lane, uint8_t* scratch, const CommitIn& in)
{
    const CacheDesc& c = p.c;
    const int g = c.g;
    const uint4 vnew4 = in.vnew4, knew4 = in.knew4;
    const uint2 vold = in.vold;
    // ---- V: v_new joins the ring; if the window would exceed R, its oldest token is quantised per token
    if (lane < kD / 8)                                                                  // window rows are unit-swizzled (win_unit)
        reinterpret_cast<uint4*>(c.v_res + (int64_t)u * c.v_res_cap * kD)[win_unit((s.vhead + s.L) % c.v_res_cap, lane)] = vnew4;
    if (s.L + 1 > c.R) {
        constexpr int F = 16 / VB, kSlabRows = 16 * F, kSlabs = 128 / kSlabRows;
        const float maxq = (float)((1 << VB) - 1);
        const int bb = lay_block_bytes(VB, g);
        uint8_t* blk = c.v_store + ((int64_t)u * c.v_cap_blocks + s.tv / kBlockTokens) * bb;
        const int inner = s.tv % kBlockTokens;
        const uint2 raw = vold;                                                         // 4 channels per lane
        const __half2* rh = reinterpret_cast<const __half2*>(&raw);
        const float2 x01 = __half22float2(rh[0]), x23 = __half22float2(rh[1]);
        const float x[4] = {x01.x, x01.y, x23.x, x23.y};
        float mnf = fminf(fminf(x[0], x[1]), fminf(x[2], x[3])), mxf = fmaxf(fmaxf(x[0], x[1]), fmaxf(x[2], x[3]));
        const int lpg = g / 4;                                                          // lanes per group
        for (int o = 1; o < lpg; o <<= 1) {
            mnf = fminf(mnf, __shfl_xor_sync(0xffffffffu, mnf, o));
            mxf = fmaxf(mxf, __shfl_xor_sync(0xffffffffu, mxf, o));
        }
        const __half d16 = __float2half_rn(mxf - mnf);
        const __half sc = __float2half_rn(__fdiv_rn(__half2float(d16), maxq));
        const float scf = __half2float(sc), rcp = __frcp_rn(scf);
        uint32_t four = 0;
        #pragma unroll
        for (int e = 0; e < 4; ++e) four |= (uint32_t)__float2int_rn(q_code(x[e], mnf, scf, rcp, maxq)) << (8 * e);
        __syncwarp();
        reinterpret_cast<uint32_t*>(scratch)[lane] = four;                              // codes[channel] as bytes
        if (lane % lpg == 0) {
            *reinterpret_cast<__half*>(blk + lay_scale_off(VB, g, inner, lane / lpg)) = sc;
            *reinterpret_cast<__half*>(blk + lay_zero_off(VB, g, inner, lane / lpg)) = __float2half_rn(mnf);
        }
        __syncwarp();
        if (lane < kSlabs * 16) {                                                       // one 16-bit half-word per lane
            const int sl = lane >> 4, row = lane & 15;
            uint32_t hw = 0;
            #pragma unroll
            for (int j = 0; j < F; ++j) hw |= (uint32_t)scratch[sl * kSlabRows + 16 * j + row] << (VB * j);
            *reinterpret_cast<uint16_t*>(blk + lay_word_off(VB, inner, sl * kSlabRows + row) + 2 * (inner & 1)) = (uint16_t)hw;
        }
        __syncwarp();
    }
    // ---- K: k_new joins the window.  (When it COMPLETES the window, r + 1 == R, the whole window is quantised instead:
    // k_flush_slice below, spread over all warps of the p.V kernel.)
    if (s.r + 1 < c.R) {
        if (lane >= 16) reinterpret_cast<uint4*>(c.k_res + (int64_t)u * c.R * kD)[win_unit(s.r, lane - 16)] = knew4;
    }
}

// ------------------------------------------------------------------------------------------------
// K flush (models/llama_kivi.py:343-356), once per R steps: the R window tokens (R - 1 rows of the fp16 window + k_new) of
// a unit are quantised per channel in groups of g tokens, straight into the fragment words of the K store.  It depends on
// nothing the attention computes and touches nothing the attention reads (blocks past tk, meta of new groups), so the
// p.V kernel does it up front, while it would otherwise wait for the q.K^T kernel to drain, spread over ALL its warps:
// slice (unit, q) = the channel pairs (8 cu + 2q, + 1), cu = 0..15, of one unit.  lane = (hw, cu): token parity hw = lane >> 4.
// A lane owns whole 32-bit words of the destination block (its channel pair, rows 2m + hw of a slab, all their fields):
// assembled in registers, stored once per slab, read-modify-write only when R < 128 leaves other tokens' fields in the word.
// (Done by the last-arriving warp of each unit at the tail of its range, the flush cost 3.8 ms per flush step at cfg 2.)
// ------------------------------------------------------------------------------------------------
template <int KB>
__device__ __noinline__ void k_flush_slice(const AttnParams& p, const Sched& s, int u, int q, int lane)
{
    const CacheDesc& c = p.c;
    const int g = c.g;
    constexpr int F = 16 / KB, kSlabRows = 16 * F, kSlabs = 128 / kSlabRows;
    const float maxq = (float)((1 << KB) - 1);
    const int bb = lay_block_bytes(KB, g);
    uint8_t* ub = c.k_store + (int64_t)u * c.k_cap_blocks * bb;
    const __half* win = c.k_res + (int64_t)u * c.R * kD;
    const __half* knew = p.k_new + (int64_t)u * kD;
    const int nblk = max(1, c.R / kBlockTokens);                                        // R in {32, 64, 128, 256}
    const int cnt = min(c.R, kBlockTokens);                                             // flushed tokens per destination block
    const int hw = lane >> 4, cu = lane & 15;
    auto row2 = [&](int t) -> __half2 {                                                 // window token t, channels 8 cu + 2q, + 1
        return t < c.R - 1 ? u32_as_h2(__ldcg(reinterpret_cast<const uint32_t*>(win + (int64_t)t * kD + ((cu ^ (t & 7)) << 3)) + q))
                           : u32_as_h2(__ldg(reinterpret_cast<const uint32_t*>(knew + 8 * cu) + q));
    };
    #pragma unroll 1
    for (int bi = 0; bi < nblk; ++bi) {
        const int tb = s.tk + bi * kBlockTokens;                                        // first flushed token of this block
        const int o0 = tb % kBlockTokens;                                               // its outer index (multiple of R)
        uint8_t* blk = ub + (int64_t)(tb / kBlockTokens) * bb;
        const bool partial = cnt < kBlockTokens;                                        // other fields of the words are live data
        // word m of slab sl: inner pair 8 cu + 2q (+1), row 2m + hw   (kivi_decode.cuh: lane' = (row & 7) * 4 + q, r = 2 (cu & 1) + (row >> 3))
        uint32_t* wbase = reinterpret_cast<uint32_t*>(blk) + (cu >> 1) * kSlabs * 128 + (cu & 1) * 2 + q * 4;
        uint32_t words[8];
        int cur_sl = -1;
        #pragma unroll 1
        for (int gl = 0; gl < cnt / g; ++gl) {                                          // groups landing in this block
            const int tl0 = bi * kBlockTokens + gl * g;                                 // first token of the group within the window
            float mn0 = INFINITY, mx0 = -INFINITY, mn1 = INFINITY, mx1 = -INFINITY;
            #pragma unroll 1
            for (int i0 = 0; i0 < g; i0 += 16) {                                        // 8 rows of this parity per pass (independent loads)
                __half2 v[8];
                #pragma unroll
                for (int m = 0; m < 8; ++m) v[m] = row2(tl0 + i0 + 2 * m + hw);
                #pragma unroll
                for (int m = 0; m < 8; ++m) {
                    const float2 f = __half22float2(v[m]);
                    mn0 = fminf(mn0, f.x); mx0 = fmaxf(mx0, f.x);
                    mn1 = fminf(mn1, f.y); mx1 = fmaxf(mx1, f.y);
                }
            }
            mn0 = fminf(mn0, __shfl_xor_sync(0xffffffffu, mn0, 16)); mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 16));   // the other token parity
            mn1 = fminf(mn1, __shfl_xor_sync(0xffffffffu, mn1, 16)); mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 16));
            const __half sc0 = __float2half_rn(__fdiv_rn(__half2float(__float2half_rn(mx0 - mn0)), maxq));
            const __half sc1 = __float2half_rn(__fdiv_rn(__half2float(__float2half_rn(mx1 - mn1)), maxq));
            const float scf0 = __half2float(sc0), scf1 = __half2float(sc1), rcp0 = __frcp_rn(scf0), rcp1 = __frcp_rn(scf1);
            const int og = o0 + gl * g;                                                 // outer index of the group's first token
            if (hw == 0) {                                                              // meta entry half: { z, z', s, s' } of the pair
                __align__(8) __half mz[4] = {__float2half_rn(mn0), __float2half_rn(mn1), sc0, sc1};
                *reinterpret_cast<uint2*>(blk + lay_zero_off(KB, g, 8 * cu + 2 * q, og / g)) = *reinterpret_cast<const uint2*>(mz);
            }
            #pragma unroll 1
            for (int q16 = 0; q16 < g / 16; ++q16) {
                const int o = og + 16 * q16;                                            // outer index of row 0 of this 16-token chunk
                const int sl = o / kSlabRows, j = (o % kSlabRows) / 16;
                if (sl != cur_sl) {
                    if (cur_sl >= 0) {
                        #pragma unroll
                        for (int m = 0; m < 8; ++m) wbase[cur_sl * 128 + ((2 * m + hw) & 7) * 16 + ((2 * m + hw) >> 3)] = words[m];
                    }
                    cur_sl = sl;
                    #pragma unroll
                    for (int m = 0; m < 8; ++m) words[m] = partial ? wbase[sl * 128 + ((2 * m + hw) & 7) * 16 + ((2 * m + hw) >> 3)] : 0u;
                }
                const uint32_t keep = ~((((1u << KB) - 1u) * 0x00010001u) << (KB * j));
                __half2 v[8];
                #pragma unroll
                for (int m = 0; m < 8; ++m) v[m] = row2(tl0 + 16 * q16 + 2 * m + hw);
                #pragma unroll
                for (int m = 0; m < 8; ++m) {
                    const float2 f = __half22float2(v[m]);
                    const uint32_t c0 = (uint32_t)__float2int_rn(q_code(f.x, mn0, scf0, rcp0, maxq));
                    const uint32_t c1 = (uint32_t)__float2int_rn(q_code(f.y, mn1, scf1, rcp1, maxq));
                    words[m] = (words[m] & keep) | ((c0 | (c1 << 16)) << (KB * j));
                }
            }
        }
        if (cur_sl >= 0) {
            #pragma unroll
            for (int m = 0; m < 8; ++m) wbase[cur_sl * 128 + ((2 * m + hw) & 7) * 16 + ((2 * m + hw) >> 3)] = words[m];
        }
    }
}

// fp32 softmax statistics of up to 32 * N values held by the warp (v < -60000 marks "no value")
__device__ __forceinline__ void warp_max_sum(float mx, float sm, float& M, float& S) {
    // (max, sum) pairs combined over the lanes
    #pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        const float mo = __shfl_xor_sync(0xffffffffu, mx, o), so = __shfl_xor_sync(0xffffffffu, sm, o);
        const float mn = fmaxf(mx, mo);
        sm = (mx == -INFINITY ? 0.f : sm * fast_exp(mx - mn)) + (mo == -INFINITY ? 0.f : so * fast_exp(mo - mn));
        mx = mn;
    }
    M = mx; S = sm;
}

// add the mask (models/llama_kivi.py:369-372) to a scaled fp16 logit
__device__ __forceinline__ __half apply_mask(__half v, const __half* mask, int64_t idx) {
    v = __hadd_rn(v, mask[idx]);
    if (__half2float(v) < -65504.f) v = __float2half_rn(-65504.f);
    return v;
}
// a left-padding position: apply_mask's arithmetic with the mask value finfo(fp16).min, so that probabilities and outputs are
// bit-identical to the additive-mask call with the equivalent mask
__device__ __forceinline__ __half apply_pad(__half v) {
    v = __hadd_rn(v, __float2half_rn(-65504.f));
    if (__half2float(v) < -65504.f) v = __float2half_rn(-65504.f);
    return v;
}

// ------------------------------------------------------------------------------------------------
// work split: the (unit, item) sequence of the whole job -- per unit: n_b packed blocks, n_w fp16 window items, the new
// token -- is cut into one contiguous range per warp of equal COST.  Costs are small integers per item kind; the first item of
// a unit may also carry the cost of a (warp, unit) visit (statistics / partial record / arrival).
//   key(pos)  = cost of everything before position pos = unit * Cu + kj(j)            (exclusive prefix, non-decreasing)
//   owner(pos) = floor(key(pos) * W / Ctot);   lo(w) = min{pos : key(pos) >= ceil(w * Ctot / W)}
// W is capped at Ctot / (largest item cost), so every range is non-empty, and a unit meets at most ceil(W / n_units) + 1
// ranges (the bound the workspace slots are sized for).
// DEFAULT: every item costs 1 (equal item counts).  A model fitted to the per-warp timeline of the cfg-2 layer (tools/timeline.py:
// q.K^T window item 0.7, new token 0.1, visit 0.6 blocks; p.V 0.4 / 1.2 / 1.2) does flatten the MODELLED cost -- the q.K^T
// lifetime spread drops from 2.1 to 1.2 us -- but the kernels get slower (cfg 2 +2 %, cfg 3 +7 %, profiles/r02_range_costs.txt):
// the tail is set by a few outlier warps (finalisations, L2-far SMs), not by the composition of the ranges.  -DKIVI_UNIFORM_RANGES=0
// builds the weighted split.
// ------------------------------------------------------------------------------------------------
#ifndef KIVI_UNIFORM_RANGES
#define KIVI_UNIFORM_RANGES 1
#endif
struct CostQK { static constexpr unsigned cb = KIVI_UNIFORM_RANGES ? 1 : 16, cw = KIVI_UNIFORM_RANGES ? 1 : 10,
                                          cn = KIVI_UNIFORM_RANGES ? 1 : 2, cv = KIVI_UNIFORM_RANGES ? 0 : 12; };
struct CostSV { static constexpr unsigned cb = KIVI_UNIFORM_RANGES ? 1 : 16, cw = KIVI_UNIFORM_RANGES ? 1 : 3,
                                          cn = KIVI_UNIFORM_RANGES ? 1 : 12, cv = KIVI_UNIFORM_RANGES ? 0 : 35; };

template <class C>
struct Ranges {
    int n_b, n_w, per_unit;
    unsigned Cu, W; unsigned long long Ctot; int small;
    // a plain struct: the kernels keep ONE copy per CTA in shared memory (its ~8 words would otherwise stay live in registers
    // across the block loops; they are read once per (warp, unit) visit)
    __host__ __device__ __forceinline__ void init(int n_units, int nb, int nw, long long w_cap) {
        n_b = nb; n_w = nw; per_unit = nb + nw + 1;
        Cu = C::cv + (unsigned)nb * C::cb + (unsigned)nw * C::cw + C::cn;
        Ctot = (unsigned long long)n_units * Cu;
        constexpr unsigned cmax = C::cv + (C::cb > C::cw ? (C::cb > C::cn ? C::cb : C::cn) : (C::cw > C::cn ? C::cw : C::cn));
        const unsigned long long n_items = (unsigned long long)n_units * per_unit;
        unsigned long long w = (unsigned long long)w_cap;
        w = w < Ctot / cmax ? w : Ctot / cmax;
        w = w < n_items ? w : n_items;
        W = (unsigned)(w < 1 ? 1 : w);
        small = (Ctot + Cu) * W < (1ull << 32) ? 1 : 0;
    }
    __host__ __device__ __forceinline__ unsigned kj(int j) const {                    // cost of items 0 .. j-1 of a unit
        if (j <= 0) return 0u;
        const int jb = min(j, n_b), jw = min(max(j - n_b, 0), n_w);
        return C::cv + (unsigned)jb * C::cb + (unsigned)jw * C::cw + (j > n_b + n_w ? C::cn : 0u);
    }
    __host__ __device__ __forceinline__ int owner(int unit, int j) const {
        if (small) return (int)(((unsigned)unit * Cu + kj(j)) * W / (unsigned)Ctot);
        return (int)(((unsigned long long)unit * Cu + kj(j)) * W / Ctot);
    }
    __host__ __device__ __forceinline__ void lo(int w, int& unit, int& j) const {     // first position of range w (w == W: the end)
        unsigned long long x;
        if (small) x = ((unsigned)w * (unsigned)Ctot + W - 1u) / W;
        else x = ((unsigned long long)w * Ctot + W - 1ull) / W;
        unit = small ? (int)((unsigned)x / Cu) : (int)(x / Cu);
        const unsigned rem = (unsigned)(x - (unsigned long long)unit * Cu);
        if (rem == 0u) { j = 0; return; }
        if (rem <= C::cv) j = 1;
        else {
            const unsigned r = rem - C::cv;
            if (r <= (unsigned)n_b * C::cb) j = (int)((r + C::cb - 1u) / C::cb);
            else if (r <= (unsigned)n_b * C::cb + (unsigned)n_w * C::cw) j = n_b + (int)((r - (unsigned)n_b * C::cb + C::cw - 1u) / C::cw);
            else j = per_unit;
        }
        if (j >= per_unit) { j = 0; ++unit; }
    }
};

struct Cursor {                         // (unit, pseudo-block, half) position of a warp in its range
    int unit, j, half, left;            // left = pseudo-blocks remaining in the range (including j)
};

// exp(x - m) with the subtraction folded into the multiply: ex2.approx(fma(x, log2 e, nml)), nml = -m * log2 e (one FFMA + MUFU)
#ifndef KIVI_EXP_FMA
#define KIVI_EXP_FMA 1
#endif
constexpr float kLog2e = 1.4426950408889634f;
__device__ __forceinline__ float fast_exp_sub(float x, float m, float nml) {
#if KIVI_EXP_FMA
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(fmaf(x, kLog2e, nml)));
    (void)m;
    return y;
#else
    (void)nml;
    return fast_exp(x - m);
#endif
}

// online softmax statistics: fold the values x[0..n) (any of them may be -inf = "no value") into (m, s)
template <int N_>
__device__ __forceinline__ void fold_stats(float& m, float& s, const float (&x)[N_]) {
    float mn = m;
    #pragma unroll
    for (int e = 0; e < N_; ++e) mn = fmaxf(mn, x[e]);
    if (mn != -INFINITY) {
        float acc = s * fast_exp(m - mn);                 // m == -inf -> s * 0
        const float nml = -mn * kLog2e;
        #pragma unroll
        for (int e = 0; e < N_; ++e) acc += fast_exp_sub(x[e], mn, nml);     // x = -inf ("no value") -> 0
        m = mn; s = acc;
    }
}

// ------------------------------------------------------------------------------------------------
// q . K^T  (+ scale, mask, per-range softmax statistics)
// ------------------------------------------------------------------------------------------------
template <int KB, int GS>
__device__ __forceinline__ void qk_issue_next(Pipe& pp, Cursor& cur, const AttnParams& p, const Sched& s,
                                              int lane, uint64_t pol)
{
    const CacheDesc& c = p.c;
    if (cur.left > 0 && cur.j == s.ipu - 1) {                     // the new token needs no load
        cur.j = 0; ++cur.unit; --cur.left;
    }
    if (cur.left <= 0) return;
    if (lane == 0) {
        const int u = p.hchunks == 1 ? cur.unit : cur.unit / p.hchunks;
        uint8_t* dst = pp.prod();
        uint64_t* bar = pp.prod_bar();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (cur.j < s.n_kb) {
            constexpr int cb = kHalfChunks * Lay<KB>::kChunkBytes;    // codes of a stage-item
            const int mb = lay_meta_bytes(GS) / kParts;
            const uint8_t* blk = c.k_store + ((int64_t)u * c.k_cap_blocks + cur.j) * lay_block_bytes(KB, GS);
            mbar_expect_tx(bar, (uint32_t)(cb + mb));
            if (kParts == 1) {
                bulk_g2s(dst, blk, (uint32_t)(cb + mb), bar, pol);    // codes and meta are contiguous: one copy
            } else {
                bulk_g2s(dst, blk + cur.half * cb, cb, bar, pol);
                bulk_g2s(dst + cb, blk + kParts * cb + cur.half * mb, (uint32_t)mb, bar, pol);
            }
        } else {
            const int t0 = (cur.j - s.n_kb) * kResTile, nt = min(kResTile, s.r - t0);
            mbar_expect_tx(bar, (uint32_t)(nt * kD * 2));
            bulk_g2s(dst, c.k_res + ((int64_t)u * c.R + t0) * kD, (uint32_t)(nt * kD * 2), bar, pol);
        }
    }
    pp.push();
    if (cur.j < s.n_kb && cur.half + 1 < kParts) { ++cur.half; return; }
    cur.half = 0;
    --cur.left;
    if (++cur.j == s.ipu) { cur.j = 0; ++cur.unit; }
}

// PAD: p.seq_start is set (left-padded batch).  A compile-time flag, so that the unpadded instantiations compile to the code
// they had without padding support (the 4-bit G = 4 kernels run 12 warps at ~160 registers and have no room to spare).
template <int KB, int G, int GS, int CW, bool PAD>
__global__ void __launch_bounds__(CW * 32, KIVI_MINB)
qk_kernel(const KIVI_PARAM_QUAL AttnParams p)
{
    constexpr int kCW = CW, kThreads = CW * 32;                              // warps / threads of this instantiation
    extern __shared__ __align__(128) uint8_t smem[];
    const CacheDesc& c = p.c;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int t4 = lane & 3;
    const int n_stages = kCW * p.spw;
    uint64_t* full_all = reinterpret_cast<uint64_t*>(smem + (size_t)n_stages * p.stage_bytes);
    uint8_t* ptr = smem + (((size_t)n_stages * (p.stage_bytes + 8) + 127) & ~(size_t)127);
    uint2* q2 = reinterpret_cast<uint2*>(ptr) + warp * (G * 32);             // per warp: [G][8 chunks][4 t] half2 pairs
    float* qlin = reinterpret_cast<float*>(ptr + kCW * G * 32 * 8) + warp * (G * kD);   // per warp: [G][128] fp32

    __shared__ Ranges<CostQK> rg_sh;                                         // items of the whole job over the range owners
    const Sched s = make_sched(c);
    if (tid < n_stages) { mbar_init(&full_all[tid], 1); mbar_fence_init(); } // one stage barrier per thread, the work split beside them
    if (tid == kThreads - 1) rg_sh.init(p.n_units, s.n_kb, s.n_kr, p.nw_eff);
    __syncthreads();                                                         // the only CTA barrier: mbarrier init, work split
    pdl_trigger();                                                           // the p.V kernel may start its prologue

    const uint64_t pol = KIVI_EVICT_FIRST ? policy_evict_first() : policy_evict_last();
    const int gw = blockIdx.x * kCW + warp;
    if (!sched_ok(s, c, p.max_kv_len)) { if (gw == 0 && lane == 0) c.state[6] = KIVI_STATE_ERR_CAPACITY; return; }
    KIVI_TL(0, gw, 0);
    const Ranges<CostQK>& rg = rg_sh;
    // a warp without a range still waits for the predecessor grid: a CTA leaves (and hands its SM to a p.V CTA, which reads
    // k_new for the K flush before its own wait) only when the kernel that produced q / k_new / v_new has completed
    if (gw >= (int)rg.W) { pdl_wait(); return; }
    int u_lo, j_lo, u_hi, j_hi;
    rg.lo(gw, u_lo, j_lo); rg.lo(gw + 1, u_hi, j_hi);
    const int n_mine = (u_hi - u_lo) * s.ipu + (j_hi - j_lo);
    Pipe pp;
    pp.init(smem + (size_t)warp * p.spw * p.stage_bytes, full_all + warp * p.spw, p.spw, p.stage_bytes);
    Cursor cur;
    cur.unit = u_lo; cur.j = j_lo; cur.half = 0; cur.left = n_mine;
    // ONE stage goes out before the grid-dependency wait (the packed cache does not depend on the predecessor); the others
    // follow the q fetch below: issued after all of a warp's first stages, the few q words queue behind the ~29 MB every warp
    // of the grid requests at this moment and arrive last -- 6.9 % of the kernel's warp time sat on their first use
    // (ncu source counters, profiles/r02_attention_ncu_summary.txt).
    for (int i = 0; i < (Lat<G>::q_first ? 1 : p.spw); ++i) qk_issue_next<KB, GS>(pp, cur, p, s, lane, pol);

    constexpr int NG = Cols<G, GS>::NG;
    const int ratio = c.H / c.Hkv;
    const int h_l = t4 % G;
    const bool slow = p.mask || p.dbg_logits;                                // mask / debug copies: rare, off the fast path

    int unit = u_lo, j = j_lo, left = n_mine;
    // q of a unit, fetched one unit ahead (registers): lane = (chunk, t) of the B-fragment pairs / 4 channels of the fp32 copy
    uint2 qf[G], ql[G];
    auto fetch_q = [&](int un) {
        const int u_ = p.hchunks == 1 ? un : un / p.hchunks, hc_ = p.hchunks == 1 ? 0 : un % p.hchunks;
        const int row0 = u_ * ratio + hc_ * G;
        #pragma unroll
        for (int h = 0; h < G; ++h) {
            const uint32_t* qh = reinterpret_cast<const uint32_t*>(p.q + (int64_t)(row0 + h) * kD + 16 * (lane >> 2) + 2 * (lane & 3));
            qf[h] = make_uint2(__ldg(qh), __ldg(qh + 4));
            ql[h] = __ldg(reinterpret_cast<const uint2*>(p.q + (int64_t)(row0 + h) * kD) + lane);
        }
    };
    pdl_wait();                                                              // q / k_new come from the previous kernel of the stream
    fetch_q(unit);
    if (Lat<G>::q_first)
        for (int i = 1; i < p.spw; ++i) qk_issue_next<KB, GS>(pp, cur, p, s, lane, pol);
    KIVI_TL(0, gw, 1);
    #pragma unroll 1
    while (left > 0) {
        const int u = p.hchunks == 1 ? unit : unit / p.hchunks, hc = p.hchunks == 1 ? 0 : unit % p.hchunks;
        const int b = u / c.Hkv;
        const int uq0 = u * ratio + hc * G;
        const int pad = PAD ? max(__ldg(p.seq_start + b), 0) : 0;         // positions < pad are padding (the new token never is)
        const int j_first = j;
        const int n_here = min(left, s.ipu - j);                             // this warp's pseudo-blocks of this unit

        // ---- this warp's copy of q: half2 pairs in B-fragment order, fp32 in channel order
        __syncwarp();
        #pragma unroll
        for (int h = 0; h < G; ++h) {
            q2[h * 32 + lane] = qf[h];
            const __half2* qh = reinterpret_cast<const __half2*>(&ql[h]);
            const float2 a = __half22float2(qh[0]), b2 = __half22float2(qh[1]);
            *reinterpret_cast<float4*>(qlin + h * kD + lane * 4) = make_float4(a.x, a.y, b2.x, b2.y);
        }
        __syncwarp();
        if (left > n_here) fetch_q(unit + 1);                                // the range continues into the next unit

        // lane-local online softmax statistics: (m_blk, s_blk) over the packed-block logits of head t4 % G held by this lane,
        // (m_win, s_win) over the window / new-token logits of head lane >> 2 held by this lane
        float m_blk = -INFINITY, s_blk = 0.f, m_win = -INFINITY, s_win = 0.f;

        #pragma unroll 1
        for (int k = 0; k < n_here; ++k, ++j) {
            if (j < s.n_kb) {                                                // ---- packed K block (tensor cores)
                float acc[8][4];
                float zc[4];
                if (kParts > 1) {                                            // whole-block stages start from D = A * B instead
                    #pragma unroll
                    for (int mm = 0; mm < 8; ++mm)
                        #pragma unroll
                        for (int e = 0; e < 4; ++e) acc[mm][e] = 0.f;
                    #pragma unroll
                    for (int e = 0; e < 4; ++e) zc[e] = 0.f;
                }
                #pragma unroll 1
                for (int half = 0; half < kParts; ++half) {
                    pp.wait();
                    mma_half<KB, G, GS, kParts == 1>(pp.cons(), half * kHalfChunks, [&](int cc, int h, uint32_t& xa, uint32_t& xb) {
                        const uint2 v = q2[(h * 8 + cc) * 4 + t4];
                        xa = v.x; xb = v.y;
                    }, acc, zc, lane);
                    __syncwarp();
                    pp.pop();
                    qk_issue_next<KB, GS>(pp, cur, p, s, lane, pol);
                }
                float zsel[NG];
                gather_z<G, GS>(zc, lane, zsel);
                const int64_t rowi = uq0 + h_l;
                __half* row = p.w.lg + rowi * p.w.ld + j * kBlockTokens;
                const int nvalid = s.tk - j * kBlockTokens;                  // < 128 only in the last block when R < 128
                // the lane's logits by compile-time slot; slots of MMAs this lane does not own and tokens past the packed
                // length stay -inf.  ONE arithmetic for the production and the instrumented / masked / partial-block
                // epilogues (same fold order, hence bit-identical statistics): they differ only in predicated side work.
                float x[Slots<G, GS>::k];
                #pragma unroll
                for (int e = 0; e < Slots<G, GS>::k; ++e) x[e] = -INFINITY;
                // (a block that overlaps the padding takes the predicated epilogue; the blocks after it keep the fast one)
                if (!slow && nvalid >= kBlockTokens && (!PAD || j * kBlockTokens >= pad)) {
                    finalize<KB, G, GS>(acc, zsel, lane, 1.f, [&](int slot, int o, float v) {
                        const __half hv = scale_logit(v);
                        row[o] = hv;
                        x[slot] = __half2float(hv);
                    });
                } else {
                    finalize<KB, G, GS>(acc, zsel, lane, 1.f, [&](int slot, int o, float v) {
                        if (o < nvalid) {
                            __half hv = scale_logit(v);                      // fp16 scaled (+ mask): the softmax input
                            if (p.mask) hv = apply_mask(hv, p.mask, (int64_t)b * s.T + j * kBlockTokens + o);
                            if (PAD && j * kBlockTokens + o < pad) hv = apply_pad(hv);
                            row[o] = hv;
                            if (p.dbg_logits) p.dbg_logits[rowi * p.dbg_stride + j * kBlockTokens + o] = hv;
                            x[slot] = __half2float(hv);
                        }
                    });
                }
                fold_stats(m_blk, s_blk, x);
            } else if (j < s.ipu - 1) {                                      // ---- fp16 K window item (tensor cores)
                // D[head][token] = sum_ch q_h[ch] * K[token][ch]: A = q (rows = heads, exact fp16), B = the window rows as they
                // lie in the stage ([token][channel], swizzled units -> conflict-free fragment loads), 2 tiles of 8 tokens
                const int t0 = (j - s.n_kb) * kResTile, nt = min(kResTile, s.r - t0);
                pp.wait();
                const uint8_t* st = pp.cons();
                float d0[4] = {0.f, 0.f, 0.f, 0.f}, d1[4] = {0.f, 0.f, 0.f, 0.f};
                const int g8 = lane >> 2;
                const int key = (t0 + g8) & 7;                               // swizzle key of rows g8 and g8 + 8 (t0 % 16 == 0)
                const uint8_t* r0 = st + g8 * 256 + t4 * 4, * r1 = r0 + 8 * 256;
                #pragma unroll
                for (int cc = 0; cc < 8; ++cc) {
                    uint2 qa = make_uint2(0u, 0u);
                    if (g8 < G) qa = q2[(g8 * 8 + cc) * 4 + t4];
                    const int u0 = ((2 * cc) ^ key) * 16, u1 = ((2 * cc + 1) ^ key) * 16;
                    mma_16816(d0, qa.x, 0u, qa.y, 0u, *reinterpret_cast<const uint32_t*>(r0 + u0), *reinterpret_cast<const uint32_t*>(r0 + u1));
                    mma_16816(d1, qa.x, 0u, qa.y, 0u, *reinterpret_cast<const uint32_t*>(r1 + u0), *reinterpret_cast<const uint32_t*>(r1 + u1));
                }
                __syncwarp();
                pp.pop();
                qk_issue_next<KB, GS>(pp, cur, p, s, lane, pol);
                // lane (g8 < G, t): head g8, tokens 2t, 2t+1 (tile 0) and 8+2t, 9+2t (tile 1)
                if (g8 < G) {
                    const int64_t rowi = uq0 + g8;
                    float x[4];
                    #pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int t = (e >> 1) * 8 + 2 * t4 + (e & 1);
                        x[e] = -INFINITY;
                        if (t < nt) {
                            __half hv = scale_logit(e < 2 ? d0[e] : d1[e - 2]);
                            if (p.mask) hv = apply_mask(hv, p.mask, (int64_t)b * s.T + s.tk + t0 + t);
                            if (PAD && s.tk + t0 + t < pad) hv = apply_pad(hv);   // a short prompt's padding reaches into the window
                            p.w.lg[rowi * p.w.ld + s.tk + t0 + t] = hv;
                            if (p.dbg_logits) p.dbg_logits[rowi * p.dbg_stride + s.tk + t0 + t] = hv;
                            x[e] = __half2float(hv);
                        }
                    }
                    fold_stats(m_win, s_win, x);
                }
            } else {                                                         // ---- the new token
                const uint2 kv = __ldg(reinterpret_cast<const uint2*>(p.k_new + (int64_t)u * kD) + lane);
                const __half2* kh = reinterpret_cast<const __half2*>(&kv);
                const float2 k01 = __half22float2(kh[0]), k23 = __half22float2(kh[1]);
                #pragma unroll
                for (int h = 0; h < G; ++h) {
                    const float4 qv = *reinterpret_cast<const float4*>(qlin + h * kD + lane * 4);
                    float sum = qv.x * k01.x;
                    sum = fmaf(qv.y, k01.y, sum); sum = fmaf(qv.z, k23.x, sum); sum = fmaf(qv.w, k23.y, sum);
                    sum = warp_sum(sum);
                    if (lane == 4 * h) {                                     // the lane that keeps head h's window statistics
                        __half hv = scale_logit(sum);
                        const int64_t rowi = uq0 + h;
                        if (p.mask) hv = apply_mask(hv, p.mask, (int64_t)b * s.T + s.T - 1);
                        p.w.lg[rowi * p.w.ld + s.T - 1] = hv;
                        if (p.dbg_logits) p.dbg_logits[rowi * p.dbg_stride + s.T - 1] = hv;
                        const float x1[1] = {__half2float(hv)};
                        fold_stats(m_win, s_win, x1);
                    }
                }
            }
        }

        // ---- this range's statistics of the unit, per head: slot = index of this warp among the unit's range owners
        const int w_first = rg.owner(unit, 0);
        #pragma unroll
        for (int h = 0; h < G; ++h) {
            float m = -INFINITY, sm = 0.f;
            if ((lane >> 2) == h) { m = m_win; sm = s_win; }
            if (h_l == h && m_blk != -INFINITY) {
                const float mn = fmaxf(m, m_blk);
                sm = (m == -INFINITY ? 0.f : sm * fast_exp(m - mn)) + s_blk * fast_exp(m_blk - mn);
                m = mn;
            }
            float M, S;
            warp_max_sum(m, sm, M, S);
            if (lane == 0) p.w.stats[(int64_t)(uq0 + h) * p.w.stat_cap + (gw - w_first)] = make_float2(M, S);
        }
#if KIVI_UNIT_FLAGS
        // publish: this range's logits (all lanes) and statistics of the unit happen-before the counter increment
        __syncwarp();
        if (lane == 0) asm volatile("red.release.gpu.global.add.s32 [%0], 1;" ::"l"(p.w.ready + unit) : "memory");
#endif
        (void)j_first;
        left -= n_here;
        if (j == s.ipu) { j = 0; ++unit; }
    }
    KIVI_TL(0, gw, 2);
#if KIVI_COMMIT_IN_QK && KIVI_EARLY_COMMIT
    // The units' cache updates (models/llama_kivi.py:343-356 without the flush, :386-399): they read k_new / v_new / the oldest
    // V window token and write only what no kernel of this step reads (the free ring slot, K window row r, token tv of the V
    // store, whose probability the p.V block loop forces to zero), so any warp may do any unit at any time after the
    // predecessor grid has completed.  A warp that has finished its range draws units from a device counter until none is
    // left: the early finishers absorb the work in the time they would wait for the stragglers of the grid, and every unit is
    // updated before the grid completes.  Which warp updates which unit does not change a single bit of the result.
    {
        const int nu = c.B * c.Hkv;
        uint8_t* scratch = reinterpret_cast<uint8_t*>(qlin);                 // this warp's 512 G bytes: q is no longer needed
        #pragma unroll 1
        for (;;) {
            int t = 0;
            if (lane == 0) t = atomicAdd(p.w.ticket, 1);
            t = __shfl_sync(0xffffffffu, t, 0);
            if (t >= nu) break;
            if (c.v_bits == 2) commit_unit<KB, 2>(p, s, t, lane, scratch, commit_fetch(p, s, t, lane));
            else commit_unit<KB, 4>(p, s, t, lane, scratch, commit_fetch(p, s, t, lane));
        }
    }
#endif
#if KIVI_PREFETCH_SV
    // This warp is done; its CTA (and the SM) stays until the slowest of its 16 warps is, and the p.V grid cannot start before
    // the whole q.K^T grid has drained.  The first packed V items of the p.V range with the same index (the p.V kernel's own
    // split, recomputed here) are requested into L2 now: HBM has spare bandwidth in this kernel's tail, and the p.V kernel's
    // first stages -- ~29 MB requested by every warp at the same moment -- then come from L2.  A hint only: no result depends on it.
    {
        Ranges<CostSV> rs;
        rs.init(p.n_units, s.n_vb, s.n_vr, p.nw_eff);
        if (gw < (int)rs.W) {
            int pu, pj;
            rs.lo(gw, pu, pj);
            #pragma unroll 1
            for (int i = 0; i < KIVI_PREFETCH_SV && pu < p.n_units; ++i) {
                if (pj < s.n_vb) {
                    if (lane == 0) {
                        const int u_ = p.hchunks == 1 ? pu : pu / p.hchunks;
                        bulk_prefetch_l2(c.v_store + ((int64_t)u_ * c.v_cap_blocks + pj) * lay_block_bytes(c.v_bits, GS),
                                         (uint32_t)lay_block_bytes(c.v_bits, GS));
                    }
                    ++pj;
                } else { pj = 0; ++pu; }                                    // window items / new token: small, skipped
            }
        }
    }
#endif
    KIVI_TL(0, gw, 3);
}

// ------------------------------------------------------------------------------------------------
// p . V  (+ softmax normalisation, output, cache update)
// ------------------------------------------------------------------------------------------------
// wait until every q.K^T range of unit `un` has published its logits and statistics (all lanes call; lane 0 spins)
__device__ __forceinline__ void wait_unit_ready(const AttnParams& p, const Sched& s, const Ranges<CostQK>& rq, int un, int lane)
{
#if KIVI_UNIT_FLAGS
    if (lane == 0) {
        const int need = rq.owner(un, s.ipu - 1) - rq.owner(un, 0) + 1;
        int have;
        do {
            asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(have) : "l"(p.w.ready + un) : "memory");
            if (have < need) __nanosleep(40);
        } while (have < need);
        asm volatile("fence.proxy.async;" ::: "memory");          // the bulk copies (async proxy) that follow read what was just acquired
    }
    __syncwarp();
#endif
}

template <int VB, int G, int GS>
__device__ __forceinline__ void sv_issue_next(Pipe& pp, Cursor& cur, const AttnParams& p, const Sched& s,
                                              int ratio, int lane, uint64_t pol, const Ranges<CostQK>& rq, int& ready_unit)
{
    const CacheDesc& c = p.c;
    if (cur.left > 0 && cur.j == s.bpu - 1) {                     // the new token needs no load
        cur.j = 0; ++cur.unit; --cur.left;
    }
    if (cur.left <= 0) return;
    if (cur.unit != ready_unit) { wait_unit_ready(p, s, rq, cur.unit, lane); ready_unit = cur.unit; }
    if (lane == 0) {
        const int u = p.hchunks == 1 ? cur.unit : cur.unit / p.hchunks, hc = p.hchunks == 1 ? 0 : cur.unit % p.hchunks;
        uint8_t* dst = pp.prod();
        uint64_t* bar = pp.prod_bar();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (cur.j < s.n_vb) {
            constexpr int cb = kHalfChunks * Lay<VB>::kChunkBytes;    // codes of a stage-item
            const int mb = lay_meta_bytes(GS) / kParts;
            const uint8_t* blk = c.v_store + ((int64_t)u * c.v_cap_blocks + cur.j) * lay_block_bytes(VB, GS);
            mbar_expect_tx(bar, (uint32_t)(cb + mb + G * kPartTokens * 2));
            if (kParts == 1) {
                bulk_g2s(dst, blk, (uint32_t)(cb + mb), bar, pol);    // codes and meta are contiguous: one copy
            } else {
                bulk_g2s(dst, blk + cur.half * cb, cb, bar, pol);
                bulk_g2s(dst + cb, blk + kParts * cb + cur.half * mb, (uint32_t)mb, bar, pol);
            }
            const int uq0 = u * ratio + hc * G;
            for (int h = 0; h < G; ++h)                               // the logits of the item's tokens (workspace rows)
                bulk_g2s(dst + cb + mb + h * kPartTokens * 2,
                         p.w.lg + (int64_t)(uq0 + h) * p.w.ld + cur.j * kBlockTokens + cur.half * kPartTokens,
                         kPartTokens * 2, bar, pol);
        } else {
            const int i = cur.j - s.n_vb;
            int slot0, nt;
            if (i < s.vr1) { const int t0 = i * kResTile; slot0 = s.vhead + t0; nt = min(kResTile, s.seg1 - t0); }
            else { const int t0 = (i - s.vr1) * kResTile; slot0 = t0; nt = min(kResTile, s.L - s.seg1 - t0); }
            if (Lat<G>::win_bulk && p.spw >= 2) {
                // + the item's logits: 48 bytes from the 16-byte boundary at or below logit (tv + l0) of every head's workspace
                // row (rows are 256-byte aligned and padded by 128 entries), behind the 16 window rows of the stage
                mbar_expect_tx(bar, (uint32_t)(nt * kD * 2 + G * 48));
                bulk_g2s(dst, c.v_res + ((int64_t)u * c.v_res_cap + slot0) * kD, (uint32_t)(nt * kD * 2), bar, pol);
                const int l0 = i < s.vr1 ? i * kResTile : s.seg1 + (i - s.vr1) * kResTile;
                const int uq0 = u * ratio + hc * G;
                for (int h = 0; h < G; ++h) {
                    const int64_t e0 = ((int64_t)(uq0 + h) * p.w.ld + s.tv + l0) & ~(int64_t)7;
                    bulk_g2s(dst + kResBytes + h * 64, p.w.lg + e0, 48u, bar, pol);
                }
            } else {
                mbar_expect_tx(bar, (uint32_t)(nt * kD * 2));
                bulk_g2s(dst, c.v_res + ((int64_t)u * c.v_res_cap + slot0) * kD, (uint32_t)(nt * kD * 2), bar, pol);
            }
        }
    }
    pp.push();
    if (cur.j < s.n_vb && cur.half + 1 < kParts) { ++cur.half; return; }
    cur.half = 0;
    --cur.left;
    if (++cur.j == s.bpu) { cur.j = 0; ++cur.unit; }
}

// fp16 probability of a scaled logit: fp16(exp(x - M) / S)   (models/llama_kivi.py:375); rS = 1 / S
__device__ __forceinline__ float prob_f32(float x, float M, float nMl, float S, float rS) {
    const float e = fast_exp_sub(x, M, nMl);
    const float q = e * rS;
    return fmaf(fmaf(-q, S, e), rS, q);     // one Newton step on the quotient = the correctly rounded e / S
}

template <int KB, int VB, int G, int GS, int CW>
__global__ void __launch_bounds__(CW * 32, KIVI_MINB)
sv_kernel(const KIVI_PARAM_QUAL AttnParams p)
{
    constexpr int kCW = CW, kThreads = CW * 32;                              // warps / threads of this instantiation
    extern __shared__ __align__(128) uint8_t smem[];
    const CacheDesc& c = p.c;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int t4 = lane & 3;
    const int n_stages = kCW * p.spw;
    uint64_t* full_all = reinterpret_cast<uint64_t*>(smem + (size_t)n_stages * p.stage_bytes);
    uint8_t* ptr = smem + (((size_t)n_stages * (p.stage_bytes + 8) + 127) & ~(size_t)127);
    float* obuf = reinterpret_cast<float*>(ptr) + warp * (G * kD);             // per warp: [G][128] window-item outputs in channel order
    uint8_t* scratch = reinterpret_cast<uint8_t*>(obuf);                     // commit_unit scratch (128 bytes), same storage
    (void)scratch;

    __shared__ Ranges<CostSV> rg_sh;                                         // this kernel's work split
    __shared__ Ranges<CostQK> rq_sh;                                         // the q.K^T kernel's (statistics slots per unit)
    const Sched s = make_sched(c);
    if (tid < n_stages) { mbar_init(&full_all[tid], 1); mbar_fence_init(); } // one stage barrier per thread, the work splits beside them
    if (tid == kThreads - 1) rg_sh.init(p.n_units, s.n_vb, s.n_vr, p.nw_eff);
    if (tid == kThreads - 33) rq_sh.init(p.n_units, s.n_kb, s.n_kr, p.nw_eff);
    __syncthreads();                                                         // the only CTA barrier: mbarrier init, work splits

    const uint64_t pol = KIVI_EVICT_FIRST ? policy_evict_first() : policy_evict_last();
    const int gw = blockIdx.x * kCW + warp;
    if (!sched_ok(s, c, p.max_kv_len)) return;                               // the q.K^T kernel has flagged state[6]
    KIVI_TL(1, gw, 0);
    const Ranges<CostSV>& rg = rg_sh;                                        // range owners: every range is non-empty
    const Ranges<CostQK>& rq = rq_sh;                                        // the qk kernel's ranges
    if (gw >= (int)rg.W) return;
    int u_lo, j_lo, u_hi, j_hi;
    rg.lo(gw, u_lo, j_lo); rg.lo(gw + 1, u_hi, j_hi);
    const int n_mine = (u_hi - u_lo) * s.bpu + (j_hi - j_lo);
    const int ratio = c.H / c.Hkv;
    Pipe pp;
    pp.init(smem + (size_t)warp * p.spw * p.stage_bytes, full_all + warp * p.spw, p.spw, p.stage_bytes);
    Cursor cur;
    cur.unit = u_lo; cur.j = j_lo; cur.half = 0; cur.left = n_mine;
    int ready_unit = -1;                                                     // last unit whose q.K^T ranges are known to be complete
    if (s.r + 1 == c.R) {                                                    // the step that completes the K window: flush it now
        const int n_slices = 4 * c.B * c.Hkv, n_workers = (int)rg.W;
        for (int sl = gw; sl < n_slices; sl += n_workers) k_flush_slice<KB>(p, s, sl >> 2, sl & 3, lane);
    }
    // The units' cache updates (V-token pack, window appends) read k_new / v_new / the oldest window token and write only what
    // no kernel of this step reads: the free ring slot, window row r, and token tv of the V store (whose probability the block
    // loop forces to zero).  They are spread evenly over the warps.  KIVI_COMMIT_LATE = 0: before the grid-dependency wait
    // (fills the time an early CTA waits for the q.K^T grid); 1: after the warp's first stages are in flight (their round
    // trips -- dependent loads queued behind the ~29 MB of first-stage copies every warp issues at that moment -- then overlap
    // the flight of the warp's own first block instead of delaying its issue: the p90 of "first stage issued" was 5 us behind
    // the median in the per-warp timeline, and those late starters set the end of the kernel).
#if !KIVI_COMMIT_IN_QK
    auto commit_share = [&]() {
        const long long nu = (long long)c.B * c.Hkv, nwk = (long long)rg.W;
        const int u0 = (int)((gw * nu + nwk - 1) / nwk), u1 = (int)(((gw + 1) * nu + nwk - 1) / nwk);
        for (int uu = u0; uu < u1; ++uu) commit_unit<KB, VB>(p, s, uu, lane, scratch, commit_fetch(p, s, uu, lane));
    };
#endif
#if KIVI_EARLY_COMMIT && !KIVI_COMMIT_LATE && !KIVI_COMMIT_IN_QK
#if KIVI_COMMIT_ASYNC
    if (p.spw < 2) commit_share();                                           // one stage per warp: no room for the inputs to travel in
#else
    commit_share();
#endif
#endif
#if !KIVI_UNIT_FLAGS
    pdl_wait();                                                              // logits and statistics come from the q.K^T kernel
#endif
#if KIVI_COMMIT_IN_QK && KIVI_EARLY_COMMIT
    if (gw == 0 && lane == 0) *p.w.ticket = 0;                               // every draw of the q.K^T grid has completed: ready for the next call
#endif

    constexpr int NG = Cols<G, GS>::NG;
    const int h_l = t4 % G;
    constexpr int kHalfBytes = kHalfChunks * Lay<VB>::kChunkBytes + kHalfChunks * NG * 64;   // codes + meta of half a V block
    const int rec = G * 2 * kD;                                              // floats of a partial record

    int unit = u_lo, j = j_lo, left = n_mine;
    // statistics slots of a unit, fetched one unit ahead: lane i holds slot i of every head
    float2 sn[G];
    int nstat = 0;
    auto fetch_stats = [&](int un) {
        const int u_ = p.hchunks == 1 ? un : un / p.hchunks, hc_ = p.hchunks == 1 ? 0 : un % p.hchunks;
        const int row0 = u_ * ratio + hc_ * G;
        nstat = rq.owner(un, s.ipu - 1) - rq.owner(un, 0) + 1;
        if (un != ready_unit) { wait_unit_ready(p, s, rq, un, lane); ready_unit = un; }
        #pragma unroll
        for (int h = 0; h < G; ++h) {
            sn[h] = make_float2(-INFINITY, 0.f);
            if (lane < nstat) sn[h] = __ldcg(p.w.stats + (int64_t)(row0 + h) * p.w.stat_cap + lane);
        }
    };
    // the few statistics words first, THEN the bulk copies: every warp of the grid issues its first stages at this very
    // moment (~29 MB in flight), and a small load queued behind them would be the last thing to arrive
    fetch_stats(unit);
#if KIVI_COMMIT_ASYNC && KIVI_EARLY_COMMIT && !KIVI_COMMIT_LATE && !KIVI_COMMIT_IN_QK
    // The inputs of this warp's (first) cache update -- the v_new row, the k_new row, the oldest V window row: 3 x 256 bytes --
    // travel as the FIRST item of the warp's stage queue and land together with its first packed block; the update itself is
    // ~250 instructions.  Fetched with ordinary loads, the same words queued behind the ~29 MB of first-stage copies all warps
    // issue at this moment: +2.9 us on the 43 % of the warps that have a unit to update, 96 % of the latest tenth of the grid
    // (profiles/r02_timeline_commit.txt).
    const long long cnu = (long long)c.B * c.Hkv, cnw = (long long)rg.W;
    const int cu0 = (int)((gw * cnu + cnw - 1) / cnw), cu1 = (int)(((gw + 1) * cnu + cnw - 1) / cnw);
    const bool commit_async = p.spw >= 2 && cu1 > cu0;
    if (commit_async) {
        if (lane == 0) {
            uint8_t* dst = pp.prod();
            uint64_t* bar = pp.prod_bar();
            const bool vq = s.L + 1 > c.R;                                   // the window is full: its oldest token gets packed
            mbar_expect_tx(bar, vq ? 768u : 512u);
            bulk_g2s_plain(dst, p.v_new + (int64_t)cu0 * kD, 256u, bar);
            bulk_g2s_plain(dst + 256, p.k_new + (int64_t)cu0 * kD, 256u, bar);
            if (vq) bulk_g2s_plain(dst + 512, c.v_res + ((int64_t)cu0 * c.v_res_cap + s.vhead) * kD, 256u, bar);
        }
        pp.push();
    }
    for (int i = commit_async ? 1 : 0; i < p.spw; ++i) sv_issue_next<VB, G, GS>(pp, cur, p, s, ratio, lane, pol, rq, ready_unit);
    KIVI_TL(1, gw, 1);
    if (commit_async) {
        pp.wait();
        const uint8_t* st = pp.cons();
        CommitIn in;
        in.vnew4 = make_uint4(0u, 0u, 0u, 0u); in.knew4 = in.vnew4; in.vold = make_uint2(0u, 0u);
        if (lane < kD / 8) in.vnew4 = reinterpret_cast<const uint4*>(st)[lane];
        if (lane >= 16) in.knew4 = reinterpret_cast<const uint4*>(st + 256)[lane - 16];
        if (s.L + 1 > c.R) in.vold = *reinterpret_cast<const uint2*>(st + 512 + 2 * (win_off(s.vhead, lane * 4) - s.vhead * kD));
        __syncwarp();
        pp.pop();
        sv_issue_next<VB, G, GS>(pp, cur, p, s, ratio, lane, pol, rq, ready_unit);     // the freed stage takes the next item at once
        commit_unit<KB, VB>(p, s, cu0, lane, scratch, in);
        for (int uu = cu0 + 1; uu < cu1; ++uu) commit_unit<KB, VB>(p, s, uu, lane, scratch, commit_fetch(p, s, uu, lane));
    }
#else
    for (int i = 0; i < p.spw; ++i) sv_issue_next<VB, G, GS>(pp, cur, p, s, ratio, lane, pol, rq, ready_unit);
    KIVI_TL(1, gw, 1);
#if KIVI_EARLY_COMMIT && KIVI_COMMIT_LATE && !KIVI_COMMIT_IN_QK
    commit_share();
#endif
#endif
    int pend_unit = -1, pend_old = 0, pend_nparts = 0;                       // arrival whose counter value is still in flight
    constexpr bool kDefer = KIVI_DEFER_ARRIVE && G == 1;                     // (the G = 4 kernels have no registers to spare)
    int arr_unit = -1, arr_nparts = 0;                                       // record written, arrival not yet issued
    auto do_arrive = [&](int un, int np) {
        __syncwarp();
        if (lane == 0) {
#if KIVI_REL_ARRIVE
            // release only: the acquire half (an L1 invalidation waiting on the atomic's round trip, 2 % of the kernel's
            // warp time over 3328 arrivals) is needed by the ONE warp that turns out to be last, and is done there
            asm volatile("atom.add.release.gpu.global.s32 %0, [%1], 1;" : "=r"(pend_old) : "l"(p.w.count + un) : "memory");
#else
            asm volatile("atom.add.acq_rel.gpu.global.s32 %0, [%1], 1;" : "=r"(pend_old) : "l"(p.w.count + un) : "memory");
#endif
        }
        pend_unit = un; pend_nparts = np;
    };
    CommitIn pend_cin = {};
    // The last warp to arrive for a unit adds the records in range order, rounds, writes the output, updates the cache.
    auto finish_unit = [&](int un, int nparts, const CommitIn& cin) {
        const int u = p.hchunks == 1 ? un : un / p.hchunks, hc = p.hchunks == 1 ? 0 : un % p.hchunks;
        const int uq0 = u * ratio + hc * G;
#if KIVI_REL_ARRIVE
        if (nparts > 1 && lane == 0) asm volatile("fence.acq_rel.gpu;" ::: "memory");   // the last arriver acquires: the counter value it read (relaxed) + this fence
#endif
        __syncwarp();                                                        // lane 0's acquire covers the other lanes' reads
        if (nparts > 1 && lane == 0) p.w.count[un] = 0;
#if KIVI_UNIT_FLAGS
        if (lane == 0) p.w.ready[un] = 0;                                    // every p.V range of the unit has long passed its acquire
#endif
        float qs[G][4], rs[G][4];
        #pragma unroll
        for (int h = 0; h < G; ++h)
            #pragma unroll
            for (int e = 0; e < 4; ++e) { qs[h][e] = 0.f; rs[h][e] = 0.f; }
        const float* r0 = p.w.part + (int64_t)un * p.w.part_cap * rec;
        constexpr int kBatch = G == 1 ? 4 : 2;                               // records loaded per round trip (independent loads)
        #pragma unroll 1
        for (int w0 = 0; w0 < nparts; w0 += kBatch) {
            float4 a[kBatch][G], b4[kBatch][G];
            #pragma unroll
            for (int k = 0; k < kBatch; ++k)
                #pragma unroll
                for (int h = 0; h < G; ++h) {
                    a[k][h] = make_float4(0.f, 0.f, 0.f, 0.f); b4[k][h] = a[k][h];
                    if (w0 + k < nparts) {
                        a[k][h] = __ldcg(reinterpret_cast<const float4*>(r0 + (int64_t)(w0 + k) * rec + (h * 2 + 0) * kD) + lane);
                        b4[k][h] = __ldcg(reinterpret_cast<const float4*>(r0 + (int64_t)(w0 + k) * rec + (h * 2 + 1) * kD) + lane);
                    }
                }
            #pragma unroll
            for (int k = 0; k < kBatch; ++k)                                 // fixed order: the sum does not depend on who arrives last
                #pragma unroll
                for (int h = 0; h < G; ++h) {
                    qs[h][0] += a[k][h].x; qs[h][1] += a[k][h].y; qs[h][2] += a[k][h].z; qs[h][3] += a[k][h].w;
                    rs[h][0] += b4[k][h].x; rs[h][1] += b4[k][h].y; rs[h][2] += b4[k][h].z; rs[h][3] += b4[k][h].w;
                }
        }
        #pragma unroll
        for (int h = 0; h < G; ++h) {
            __align__(8) __half o4[4];
            #pragma unroll
            for (int e = 0; e < 4; ++e) {
                __half o = __float2half_rn(rs[h][e]);                                   // llama_kivi.py:380 / :384
                if (s.tv > 0) o = __hadd_rn(__float2half_rn(qs[h][e]), o);             // :382-384
                o4[e] = o;
            }
            *reinterpret_cast<uint2*>(p.out + (int64_t)(uq0 + h) * kD + lane * 4) = *reinterpret_cast<const uint2*>(o4);
        }
#if !KIVI_EARLY_COMMIT
        if (hc == 0) commit_unit<KB, VB>(p, s, u, lane, scratch, cin);
#else
        (void)u; (void)cin;
#endif
    };
    #pragma unroll 1
    while (left > 0) {
        const int u = p.hchunks == 1 ? unit : unit / p.hchunks, hc = p.hchunks == 1 ? 0 : unit % p.hchunks;
        const int uq0 = u * ratio + hc * G;
        const int n_here = min(left, s.bpu - j);                             // this warp's pseudo-blocks of this unit

        // ---- (M, S) of every head of the unit from the statistics slots of the qk ranges (identical in every warp);
        // the slots were fetched one unit ahead
        float M[G], S[G], rS[G], nMl[G];
        #pragma unroll
        for (int h = 0; h < G; ++h) {
            float mx = sn[h].x, sm = sn[h].y;
            const float2* st = p.w.stats + (int64_t)(uq0 + h) * p.w.stat_cap;
            for (int i = lane + 32; i < nstat; i += 32) {                    // more than 32 ranges on one unit: few, long units
                const float2 v = __ldcg(st + i);
                const float mn = fmaxf(mx, v.x);
                sm = (mx == -INFINITY ? 0.f : sm * fast_exp(mx - mn)) + (v.x == -INFINITY ? 0.f : v.y * fast_exp(v.x - mn));
                mx = mn;
            }
            warp_max_sum(mx, sm, M[h], S[h]);
            nMl[h] = -M[h] * kLog2e;
            rS[h] = __frcp_rn(S[h]);
        }
        if (left > n_here) fetch_stats(unit + 1);                            // the range continues into the next unit

        // packed part: the MMA accumulators live for ONE block (mma.sync accumulates with truncation: a 100-step chain
        // would bias the sum by ~100 * 2^-24 of its L1 mass); the lane's own outputs are then added, rounded to nearest,
        // to running sums over this warp's blocks of the unit
        float run[Slots<G, GS>::k];
        float orr[G][4];                                                     // window part: lane = 4 channels
        #pragma unroll
        for (int e = 0; e < Slots<G, GS>::k; ++e) run[e] = 0.f;
        #pragma unroll
        for (int h = 0; h < G; ++h)
            #pragma unroll
            for (int e = 0; e < 4; ++e) orr[h][e] = 0.f;

        #pragma unroll 1
        for (int k = 0; k < n_here; ++k, ++j) {
            if (j < s.n_vb) {                                                // ---- packed V block (tensor cores)
                float acc[8][4];
                float zc[4];
                if (kParts > 1) {
                    #pragma unroll
                    for (int mm = 0; mm < 8; ++mm)
                        #pragma unroll
                        for (int e = 0; e < 4; ++e) acc[mm][e] = 0.f;
                    #pragma unroll
                    for (int e = 0; e < 4; ++e) zc[e] = 0.f;
                }
                #pragma unroll 1
                for (int half = 0; half < kParts; ++half) {
                    const int t0 = j * kBlockTokens + half * kPartTokens, nt = s.tv - t0;   // nt >= kPartTokens except at the end of the store
                    pp.wait();
                    uint8_t* st = pp.cons();
                    __half* prob = reinterpret_cast<__half*>(st + kHalfBytes);   // [G][kPartTokens] logits -> probabilities x 2^6
                    #pragma unroll
                    for (int h = 0; h < G; ++h) {
                        #pragma unroll
                        for (int e = 0; e < kPartTokens / 64; ++e) {         // 2 tokens per lane and pass
                            const int tt = (e * 32 + lane) * 2;
                            const float2 f = __half22float2(*reinterpret_cast<const __half2*>(prob + h * kPartTokens + tt));
                            __half2 pr = __floats2half2_rn(prob_f32(f.x, M[h], nMl[h], S[h], rS[h]), prob_f32(f.y, M[h], nMl[h], S[h], rS[h]));
                            if (tt >= nt) pr = __float2half2_rn(0.f);        // tokens beyond the packed length belong to the window
                            else if (tt + 1 >= nt) pr = __halves2half2(__low2half(pr), __float2half_rn(0.f));
                            if (p.dbg_probs) {
                                if (tt < nt) p.dbg_probs[(int64_t)(uq0 + h) * p.dbg_stride + t0 + tt] = __low2half(pr);
                                if (tt + 1 < nt) p.dbg_probs[(int64_t)(uq0 + h) * p.dbg_stride + t0 + tt + 1] = __high2half(pr);
                            }
                            *reinterpret_cast<__half2*>(prob + h * kPartTokens + tt) = __hmul2(pr, __float2half2_rn(kProbScale));   // exact
                        }
                    }
                    __syncwarp();
                    mma_half<VB, G, GS, kParts == 1>(st, half * kHalfChunks, [&](int cc, int h, uint32_t& xa, uint32_t& xb) {
                        const __half* pr = prob + h * kPartTokens + 16 * (cc - half * kHalfChunks) + 2 * t4;
                        xa = *reinterpret_cast<const uint32_t*>(pr);
                        xb = *reinterpret_cast<const uint32_t*>(pr + 8);
                    }, acc, zc, lane);
                    __syncwarp();
                    pp.pop();
                    sv_issue_next<VB, G, GS>(pp, cur, p, s, ratio, lane, pol, rq, ready_unit);
                }
                float zsel[NG];
                gather_z<G, GS>(zc, lane, zsel);
                finalize<VB, G, GS>(acc, zsel, lane, 1.f, [&](int slot, int, float v) { run[slot] += v; });
            } else if (j < s.bpu - 1) {                                      // ---- fp16 V window item (tensor cores)
                // D[channel][head] = sum_tok V[tok][channel] * p_h[tok]: A = the window rows as they lie in the stage
                // ([token][channel], swizzled units), delivered transposed by ldmatrix; B = the probabilities (exact fp16)
                const int i = j - s.n_vb;
                int l0, nt, slot0;                                           // logical index / ring slot of the item's first token
                if (i < s.vr1) { l0 = i * kResTile; nt = min(kResTile, s.seg1 - l0); slot0 = s.vhead + l0; }
                else { const int tt0 = (i - s.vr1) * kResTile; l0 = s.seg1 + tt0; nt = min(kResTile, s.L - s.seg1 - tt0); slot0 = tt0; }
                // the item's probabilities: lane t < nt computes token tv + l0 + t
                const bool win_bulk = Lat<G>::win_bulk && p.spw >= 2;        // (one stage per warp: nothing is prefetched, measured slower)
                if (win_bulk) pp.wait();                                     // the logits arrive with the window rows
                uint8_t* st = pp.cons();
                float pl[G];
                #pragma unroll
                for (int h = 0; h < G; ++h) {
                    pl[h] = 0.f;
                    if (lane < nt) {
                        float x;
                        if (win_bulk) {
                            const int off = (int)(((int64_t)(uq0 + h) * p.w.ld + s.tv + l0) & 7);
                            x = __half2float(reinterpret_cast<const __half*>(st + kResBytes + h * 64)[off + lane]);
                        } else {
                            x = __half2float(__ldcg(p.w.lg + (int64_t)(uq0 + h) * p.w.ld + s.tv + l0 + lane));
                        }
                        const __half pr = __float2half_rn(prob_f32(x, M[h], nMl[h], S[h], rS[h]));
                        if (p.dbg_probs) p.dbg_probs[(int64_t)(uq0 + h) * p.dbg_stride + s.tv + l0 + lane] = pr;
                        pl[h] = __half2float(pr);
                    }
                }
                const int g8 = lane >> 2;
                uint32_t b0 = 0u, b1 = 0u;                                   // column g8 = head g8: tokens 2t, 2t+1 | 2t+8, 2t+9
                #pragma unroll
                for (int h = 0; h < G; ++h) {
                    const float p0 = __shfl_sync(0xffffffffu, pl[h], 2 * t4), p1 = __shfl_sync(0xffffffffu, pl[h], 2 * t4 + 1);
                    const float p2 = __shfl_sync(0xffffffffu, pl[h], 2 * t4 + 8), p3 = __shfl_sync(0xffffffffu, pl[h], 2 * t4 + 9);
                    if (g8 == h) { b0 = h2_as_u32(__floats2half2_rn(p0, p1)); b1 = h2_as_u32(__floats2half2_rn(p2, p3)); }
                }
                if (!win_bulk) pp.wait();
                if (nt < kResTile) {                                         // rows past the item hold stale bytes (maybe NaN patterns)
                    for (int idx = lane; idx < (kResTile - nt) * 16; idx += 32)
                        *reinterpret_cast<uint4*>(st + nt * 256 + idx * 16) = make_uint4(0u, 0u, 0u, 0u);
                    __syncwarp();
                }
                // ldmatrix: lanes 8i .. 8i+7 address the rows of matrix i = (tokens 8*(i>>1) .., channel unit 2*mt + (i&1))
                const int tr = ((lane >> 4) << 3) + (lane & 7);
                const uint8_t* rowp = st + tr * 256;
                const int key = (slot0 + tr) & 7, usel = (lane >> 3) & 1;
                float oacc[8][4];
                #pragma unroll
                for (int mt = 0; mt < 8; ++mt) {
                    #pragma unroll
                    for (int e = 0; e < 4; ++e) oacc[mt][e] = 0.f;
                    uint32_t af[4];
                    ldmatrix_x4_trans(af, rowp + (((2 * mt + usel) ^ key) << 4));
                    mma_16816(oacc[mt], af[0], af[1], af[2], af[3], b0, b1);
                }
                __syncwarp();
                pp.pop();
                sv_issue_next<VB, G, GS>(pp, cur, p, s, ratio, lane, pol, rq, ready_unit);
                // lane (g8, t): oacc[mt] = D[16mt + g8 | + 8][heads 2t, 2t+1] -> channel order through shared memory
                #pragma unroll
                for (int mt = 0; mt < 8; ++mt)
                    #pragma unroll
                    for (int e = 0; e < 2; ++e)
                        if (2 * t4 + e < G) {
                            obuf[(2 * t4 + e) * kD + 16 * mt + g8] = oacc[mt][e];
                            obuf[(2 * t4 + e) * kD + 16 * mt + g8 + 8] = oacc[mt][2 + e];
                        }
                __syncwarp();
                #pragma unroll
                for (int h = 0; h < G; ++h) {
                    const float4 v = *reinterpret_cast<const float4*>(obuf + h * kD + lane * 4);
                    orr[h][0] += v.x; orr[h][1] += v.y; orr[h][2] += v.z; orr[h][3] += v.w;
                }
                __syncwarp();
            } else {                                                         // ---- the new token (v_new)
                const uint2 vv = __ldg(reinterpret_cast<const uint2*>(p.v_new + (int64_t)u * kD) + lane);
                const __half2* vh = reinterpret_cast<const __half2*>(&vv);
                const float2 v01 = __half22float2(vh[0]), v23 = __half22float2(vh[1]);
                #pragma unroll
                for (int h = 0; h < G; ++h) {
                    const float x = __half2float(__ldcg(p.w.lg + (int64_t)(uq0 + h) * p.w.ld + s.T - 1));
                    const __half prh = __float2half_rn(prob_f32(x, M[h], nMl[h], S[h], rS[h]));
                    if (p.dbg_probs && lane == 0) p.dbg_probs[(int64_t)(uq0 + h) * p.dbg_stride + s.T - 1] = prh;
                    const float pr = __half2float(prh);
                    orr[h][0] = fmaf(pr, v01.x, orr[h][0]); orr[h][1] = fmaf(pr, v01.y, orr[h][1]);
                    orr[h][2] = fmaf(pr, v23.x, orr[h][2]); orr[h][3] = fmaf(pr, v23.y, orr[h][3]);
                }
            }
            if (kDefer && arr_unit >= 0) { do_arrive(arr_unit, arr_nparts); arr_unit = -1; }   // the previous unit's arrival, one item later
        }

        // ---- this warp's partial record of the unit: [G][packed | window][128]
        const int w_first = rg.owner(unit, 0), w_last = rg.owner(unit, s.bpu - 1);
        const int nparts = w_last - w_first + 1;
        float* recp = p.w.part + ((int64_t)unit * p.w.part_cap + (gw - w_first)) * rec;
        {
            float* rq = recp + (h_l * 2 + 0) * kD;
            walk_slots<G, GS>(run, lane, [&](int o, float v) { rq[o] = v * kProbScaleInv; });
            #pragma unroll
            for (int h = 0; h < G; ++h)
                *reinterpret_cast<float4*>(recp + (h * 2 + 1) * kD + lane * 4) = make_float4(orr[h][0], orr[h][1], orr[h][2], orr[h][3]);
        }
        // the arrival of the PREVIOUS unit has had a whole unit's time to return: finalise it if this warp was its last
        if (pend_unit >= 0 && __shfl_sync(0xffffffffu, pend_old, 0) == pend_nparts - 1) finish_unit(pend_unit, pend_nparts, pend_cin);
        pend_unit = -1;
        // the inputs of this unit's cache update travel together with the arrival below
#if !KIVI_EARLY_COMMIT
        pend_cin = commit_fetch(p, s, u, lane);
#endif
        // arrive: the records of all lanes happen-before lane 0's release (__syncwarp), and its acquire makes the records of
        // the earlier arrivals visible to a last arriver; the counter's old value is not needed before the next unit is
        // done, so its round trip to L2 is off the critical path
        if (nparts > 1) {
            // another visit follows: the arrival waits until its first item is done -- by then the record stores above have
            // landed and the release fence (7 % of the kernel's warp time when it follows the stores directly) returns at once
            if (kDefer && left > n_here) { arr_unit = unit; arr_nparts = nparts; }
            else do_arrive(unit, nparts);
        } else {
            __syncwarp();
            finish_unit(unit, 1, pend_cin);                                  // the whole unit was this warp's
        }
        left -= n_here;
        if (j == s.bpu) { j = 0; ++unit; }
    }
    KIVI_TL(1, gw, 2);
    if (pend_unit >= 0 && __shfl_sync(0xffffffffu, pend_old, 0) == pend_nparts - 1) finish_unit(pend_unit, pend_nparts, pend_cin);
    KIVI_TL(1, gw, 3);
}

// ------------------------------------------------------------------------------------------------
// host
// ------------------------------------------------------------------------------------------------
constexpr int kMaxCtasPerSm = KIVI_MINB;

// workspace carve-up (shared by kivi_decode_workspace_bytes and the launcher); negative = KIVI_ERR_* / -cudaError
static inline int64_t carve_workspace(const CacheDesc& c, int n_units, int G, int max_kv_len, void* base, Workspace* w)
{
    DeviceInfo di;
    const int drc = device_info(&di);
    if (drc) return drc < 0 ? drc : -(int64_t)drc;
    const int64_t rows = (int64_t)c.B * c.H;
    const int64_t ld = ((int64_t)max_kv_len + 16 + 127) / 128 * 128 + 128;
    const int bpu_max = cdiv(max_kv_len, kBlockTokens) + cdiv(c.R + 1, kResTile) + 4;
    const int warps = di.num_sms * kMaxCtasPerSm * kCW;                     // the largest CTA any instantiation launches
    const int part_cap = min(bpu_max, cdiv(warps, n_units) + 2);
    int64_t off = 0;
    auto take = [&](int64_t bytes) { const int64_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    const int64_t o_lg = take(rows * ld * 2);
    const int stat_cap = part_cap;                                          // one slot per qk range of a unit
    const int64_t o_st = take(rows * stat_cap * 8);
    const int64_t o_pt = take((int64_t)n_units * part_cap * G * 2 * kD * 4);
    const int64_t o_ct = take((int64_t)n_units * 4);
    const int64_t o_rd = take((int64_t)n_units * 4);
    const int64_t o_tk = take(4);
    if (w) {
        uint8_t* b = (uint8_t*)base;
        w->lg = (__half*)(b + o_lg); w->ld = ld;
        w->stats = (float2*)(b + o_st); w->stat_cap = stat_cap;
        w->part = (float*)(b + o_pt); w->part_cap = part_cap;
        w->count = (int*)(b + o_ct);
        w->ready = (int*)(b + o_rd);
        w->ticket = (int*)(b + o_tk);
    }
    return off;
}

template <int KB, int VB, int G, int GS>
static int launch_attention(AttnParams& p, bool overlap_prologue, cudaStream_t st)
{
    const CacheDesc& c = p.c;
    DeviceInfo di;
    int rc = device_info(&di);
    if (rc) return rc;
    const Tuning& tn = tuning();
    constexpr int kCW = WarpsPerCta<KB, G>::k, kThreads = kCW * 32;          // (shadows the global default)
    const int max_smem = di.max_smem_optin - 1024;                           // room for the kernels' static shared memory (work split, 128 B)
    const int half_k = kHalfChunks * Lay<KB>::kChunkBytes + lay_meta_bytes(c.g) / kParts;
    const int half_v = kHalfChunks * Lay<VB>::kChunkBytes + lay_meta_bytes(c.g) / kParts + G * kPartTokens * 2;
    const int stage = max(max(half_k, half_v), kResBytes + G * 64);           // a window item: 16 rows + 48 B of logits per head
    p.stage_bytes = (stage + 127) / 128 * 128;
    const int fixed = 512 + kCW * G * (32 * 8 + kD * 4);                     // barriers + per-warp q buffers (qk) / window outputs (sv)
    int ctas = kMaxCtasPerSm;                                                // the kernels' __launch_bounds__
    p.spw = 0;
    for (; ctas >= 1; --ctas) {                                              // most CTAs per SM that still get >= 2 stages per warp
        p.spw = min(4, (max_smem / ctas - fixed) / (kCW * p.stage_bytes));
        if (p.spw >= 2) break;
    }
    if (ctas < 1) { ctas = 1; p.spw = (max_smem - fixed) / (kCW * p.stage_bytes); }
    if (tn.ctas_per_sm >= 1 && tn.ctas_per_sm <= ctas) {                     // tuning knobs (tools/microbench.py), read once per process
        ctas = tn.ctas_per_sm;
        p.spw = min(8, (max_smem / ctas - fixed) / (kCW * p.stage_bytes));
    }
    if (tn.stages_per_warp >= 1 && tn.stages_per_warp <= p.spw) p.spw = tn.stages_per_warp;
    if (p.spw < 1) return KIVI_ERR_CAPACITY;
    const size_t smem = (size_t)kCW * p.spw * p.stage_bytes + fixed;
    auto kqk = p.seq_start ? qk_kernel<KB, G, GS, kCW, true> : qk_kernel<KB, G, GS, kCW, false>;
    auto ksv = sv_kernel<KB, VB, G, GS, kCW>;
    static std::atomic<unsigned long long> optin_qk{0}, optin_qk_pad{0}, optin_sv{0};   // per kernel instantiation, one bit per device
    rc = ensure_dynamic_smem(kqk, max_smem, di.ordinal, p.seq_start ? optin_qk_pad : optin_qk); if (rc) return rc;
    rc = ensure_dynamic_smem(ksv, max_smem, di.ordinal, optin_sv); if (rc) return rc;
    const int grid = di.num_sms * ctas;
    // range owners: at least one pseudo-block each (the kernels clamp to the number of pseudo-blocks), and never more
    // ranges per unit than the workspace has record / statistics slots: part_cap - 2 warps per unit at most
    const long long want = (long long)p.n_units * max(1, p.w.part_cap - 2);
    p.nw_eff = (int)min((long long)grid * kCW, want);
    // programmatic dependent launch: the p.V prologue (setup, cache lengths) overlaps the q.K^T tail; the q.K^T prologue
    // (setup, lengths, first K blocks in flight) overlaps the tail of the previous kernel of the stream only when the
    // caller has promised that that kernel does not write the cache (KIVI_CACHE_OVERLAP_PROLOGUE)
    const bool pdl = !tn.no_pdl;
    cudaLaunchAttribute attr_qk[1], attr_sv[1];
    attr_qk[0].id = attr_sv[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr_qk[0].val.programmaticStreamSerializationAllowed = pdl && overlap_prologue ? 1 : 0;
    attr_sv[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kThreads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cfg.attrs = attr_qk; cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kqk, p);
    if (e != cudaSuccess) return (int)e;
    rc = post_launch(); if (rc) return rc;
    cfg.attrs = attr_sv;
    e = cudaLaunchKernelEx(&cfg, ksv, p);
    if (e != cudaSuccess) return (int)e;
    return post_launch();
}

template <int KB, int VB>
static int dispatch_attention(AttnParams& p, int G, bool overlap_prologue, cudaStream_t st)
{
    #define KIVI_GS(GS_)                                                                  \
        if (p.c.g == GS_) {                                                               \
            if (G == 4) return launch_attention<KB, VB, 4, GS_>(p, overlap_prologue, st);                   \
            if (G == 2) return launch_attention<KB, VB, 2, GS_>(p, overlap_prologue, st);                   \
            return launch_attention<KB, VB, 1, GS_>(p, overlap_prologue, st);                               \
        }
    KIVI_GS(32)
    KIVI_GS(64)
    KIVI_GS(128)
    #undef KIVI_GS
    return KIVI_ERR_GROUP;
}

}  // namespace kivi
