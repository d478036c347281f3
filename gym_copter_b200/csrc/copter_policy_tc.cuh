// copter_policy_tc.cuh -- the tanh MLP policy of BASELINE.json configs[4] (O -> 64 -> 64 -> A) on the
// 5th-generation tensor cores: tcgen05.mma with the accumulators in tensor memory (TMEM).
//
// A tile is 128 envs.  Epilogue thread t owns env t of the tile AND lane t of tensor memory, so a layer is:
//   the MMA warp's elected lane issues the layer's MMAs (A = the tile's activations in shared memory,
//   B = the layer's weights in shared memory, D = 128 x 64 fp32 in TMEM)  ->  tcgen05.commit on an mbarrier
//   ->  every epilogue thread pulls ITS OWN row of D out of TMEM (tcgen05.ld 32x32b), applies tanh, rounds
//   to fp16 and writes the row back to shared memory as the next layer's A operand  ->  mbarrier arrive.
// The epilogue warps issue no MMA, no fragment loads and no bias adds (the biases ride along as one extra
// K-step: a constant A tile of ones times a B tile holding each bias split into two 16-bit halves, hi + lo,
// so the bias keeps ~16 bits).  What is left per env is 132 tanh + 66 packs + the TMEM loads; the floor is
// the MUFU pipe, and because three quarters of the issue slots and the whole FMA pipe are free here, a
// quarter of the hidden tanh are evaluated as a polynomial on the FMA pipe instead (kPolyLanes).
//
// Operand layout: the canonical K-major, no-swizzle UMMA layout -- 8-row x 16-byte "core matrices" of
// 128 contiguous bytes; core matrices adjacent in K are LBO = 128 B apart, 8-row groups SBO = (K/8) x
// 128 B apart.  A thread writing its own 128-byte activation row therefore writes eight 16-byte chunks
// 128 B apart; consecutive threads are 16 B apart inside a core matrix, so a warp's store is conflict-free.
// TMEM: one tile in flight per CTA, 64 accumulator columns (the 16 output columns of layer 3 reuse the hidden ones,
// see kColOut), so up to eight CTAs could share an SM's 512 columns -- registers and shared memory allow seven --
// and overlap one another's phases.
// Measured history and the A/B against the warp-MMA kernel (copter_policy.cuh): the comment on the kernel.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace copter {
namespace tc {

constexpr int kTile = 128, kH = 64, kK1 = 16, kN3 = 16;
// TMEM columns of a CTA: 64.  The 16 output accumulator columns of layer 3 REUSE the first columns of the hidden
// accumulator: layer 3 is issued only after every epilogue thread has pulled its layer-2 row out of TMEM (the ready
// barrier), and layer 1 of the next tile only after every thread has read its output columns.  64 columns per tile
// instead of 128 is what lets more than four CTAs share an SM's 512 columns.
constexpr uint32_t kTmemCols = 64;                  // tcgen05.alloc takes powers of two >= 32
constexpr uint32_t kColHidden = 0, kColOut = 0;
constexpr uint32_t kOnesSBO = 0;                    // the ones tile: one 8-row group, read 16 times (Smem::ones)

// element offset of (row r, column k) in a canonical K-major tile with KC = K/8 chunks per row
__device__ __forceinline__ int canon(int r, int k, int KC) { return (((r >> 3) * KC + (k >> 3)) << 6) + ((r & 7) << 3) + (k & 7); }

struct alignas(128) SlotSmem {
    // layer 2 / layer 3 activations [128 x 64]; its first 4 KB double as the layer-1 A tile (the observation rows,
    // [128 x 16]): that tile is dead once layer 1's MMAs have completed, which is before any thread writes `a`, and
    // the next tile's observation rows are written only after layer 3's MMAs -- the last readers of `a` -- completed
    __nv_bfloat16 a[kTile * kH];
    __device__ __forceinline__ __nv_bfloat16* a1() { return a; }
};
struct alignas(128) Smem {
    __nv_bfloat16 w1[kH * kK1];          // layer 1 weights  [64 x 16]  (columns OBS.. are zero, 14 / 15 carry the bias hi / lo)
    __nv_bfloat16 w2[kH * kH];           // layer 2 weights  [64 x 64]
    __nv_bfloat16 b2[kH * kK1];          // layer 2 bias step [64 x 16] (column 0 = hi, 1 = lo)
    __nv_bfloat16 w3[kN3 * kH];          // layer 3 weights  [16 x 64]  (rows ACT.. are zero)
    __nv_bfloat16 b3[kN3 * kK1];         // layer 3 bias step [16 x 16]
    // A tile of the bias steps: columns 0, 1 = 1.  All 128 rows are the same, so only ONE 8-row group is stored and
    // the descriptor's stride between row groups is 0 (kOnesSBO): 256 B instead of 4 KB, which is what lets a seventh
    // CTA fit into an SM's shared memory.
    __nv_bfloat16 ones[8 * kK1];
    SlotSmem slot;                       // the tile in flight
    uint64_t done;                       // MMA warp -> epilogue warps: the accumulator is complete (tcgen05.commit)
    uint64_t ready;                      // epilogue threads -> MMA warp: the next A tile is in shared memory (128 arrivals)
    uint64_t clc_bar[2];                 // cluster launch control: response k has landed in clc_resp[k & 1] (see next_tile)
    alignas(16) uint4 clc_resp[2];
    uint32_t tmem_base;
};

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor: canonical K-major, SWIZZLE_NONE, version 1 (sm_100)
__device__ __forceinline__ uint64_t make_desc(const void* tile, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    return (uint64_t)((smem_addr(tile) >> 4) & 0x3FFFu) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46);
}
// instruction descriptor: D = fp32, A and B of one 16-bit format, both K-major, M = 128
// The HIDDEN activations (the A operand of layers 2 and 3) are fp16, not bf16 -- three more significand bits for
// values in [-1, 1]: the error against the fp64 network halves (max 0.0046 / mean 0.0007 instead of 0.0092 / 0.0016
// on the microbenchmark's network).  A pair is two tanh.approx.f32 or two polynomials, then one cvt.rn.f16x2.f32; the
// packed `cvt.rn.f16x2.f32` + `tanh.approx.f16x2` (two issue slots per pair instead of three) was measured SLOWER
// (0.275 vs 0.267 ms, profiles/r2_sweep_policy_tc_f16.txt: the packed tanh costs the XU pipe its two slots and then
// some; the knob is removed, the last tree that has it is commit d11af01).  The observation rows (layer 1's A operand,
// unbounded magnitudes) and layer 1's weights stay bf16; the weights and bias tiles of layers 2 and 3 are fp16 as well
// (an MMA whose descriptor mixes an fp16 A with a bf16 B raises "illegal instruction" on sm_100a: measured).
// ab_bf16: format of the A and B operands (bits 7-9 and 10-12: 0 = fp16, 1 = bf16)
__host__ __device__ constexpr uint32_t make_idesc(int n, bool ab_bf16 = true) { return (1u << 4) | ((ab_bf16 ? 1u : 0u) << 7) | ((ab_bf16 ? 1u : 0u) << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTile >> 4) << 24); }

__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}"
                 :: "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate), "r"(0u) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void bar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_addr(bar)), "r"(count));
}
__device__ __forceinline__ void bar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_addr(bar)) : "memory");
}
// Waiting warps must not eat the issue slots of the working ones: a warp's TMEM lane quarter ties it to the SM
// sub-partition warp % 4, so the MMA warps of ALL resident CTAs (warp 4) sit on sub-partition 0, and a tight
// try_wait loop there starves that sub-partition's epilogue warps -- whose tiles cannot finish before they do.
// So try_wait carries a suspend-time hint: the thread sleeps in hardware until the phase completes or the hint
// expires.  (A tight try_wait loop and a loop with __nanosleep were the alternatives; the last tree that has them is
// commit d11af01.)
constexpr uint32_t kWaitHintNs = 20000;
__device__ __forceinline__ void bar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\t"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
                 "@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}" :: "r"(smem_addr(bar)), "r"(parity), "r"(kWaitHintNs) : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync()  { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem()  { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// one lane of a converged warp (the MMA warp runs its loop warp-uniformly and elects the issuing lane per instruction
// group: the descriptors then live in uniform registers instead of being moved there, R2UR, before every MMA)
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}
// Cluster launch control (sm_100): the grid holds one CTA per tile; a running CTA cancels a CTA that has not been
// launched yet and takes over its block index.  The 16-byte response lands in shared memory through an mbarrier.
// The warp scheduler favours the warps of the CTA that arrived first on an SM: with a static grid stride the first CTA
// of an SM finished its 88 tiles after 469 000 cycles and the fifth after 611 000 (the launch's duration) -- with
// stolen tiles every CTA works until the tiles run out.  (The grid-stride schedule: the last tree that has it is
// commit d11af01.)
__device__ __forceinline__ void clc_try_cancel(void* resp16, uint64_t* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], 16;" :: "r"(smem_addr(bar)) : "memory");
    asm volatile("clusterlaunchcontrol.try_cancel.async.shared::cta.mbarrier::complete_tx::bytes.b128 [%0], [%1];"
                 :: "r"(smem_addr(resp16)), "r"(smem_addr(bar)) : "memory");
}
constexpr uint32_t kNoTile = 0xFFFFFFFFu;
__device__ __forceinline__ uint32_t clc_response(const void* resp16) {      // the cancelled CTA's blockIdx.x, or kNoTile
    uint32_t ok, x;
    asm volatile("{\n\t.reg .b128 r;\n\t.reg .pred p;\n\t.reg .b64 lo, hi;\n\t.reg .b32 y, z, w;\n\t"
                 "ld.shared.v2.b64 {lo, hi}, [%2];\n\t"
                 "mov.b128 r, {lo, hi};\n\t"
                 "clusterlaunchcontrol.query_cancel.is_canceled.pred.b128 p, r;\n\t"
                 "selp.u32 %0, 1, 0, p;\n\t"
                 "mov.u32 %1, 0;\n\t"
                 "@p clusterlaunchcontrol.query_cancel.get_first_ctaid.v4.b32.b128 {%1, y, z, w}, r;\n\t}"
                 : "=r"(ok), "=r"(x) : "r"(smem_addr(resp16)) : "memory");
    return ok ? x : kNoTile;
}

// 16 consecutive fp32 columns of this thread's TMEM lane (asynchronous: tmem_wait() before the values are used)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, float (&v)[4]) {
    uint32_t r[4];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
    tmem_wait();
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = __uint_as_float(r[j]);
}

// Developer timeline (tools/microbench/policy_tc_trace.cu): clock64 stamps of a few CTAs' steady-state tiles --
// who = epilogue warp 0..3 (lane 0) or 4 = the MMA thread; event = 3 * layer + {0: woke up, 1: work done, 2: arrived / committed};
// 12 + 8 * (layer - 1) + 2 q + {0: chunk q of the hidden accumulator has landed, 1: its tanh / packs / stores are issued}.
#ifdef COPTER_POLICY_TC_TRACE
constexpr int kTraceCtas = 4, kTraceTiles = 8, kTraceFirstTile = 30, kTraceCtaStep = 211;
__device__ long long g_trace[kTraceCtas][kTraceTiles][5][32];
__device__ __forceinline__ void trace(int who, int round, int event) {
    const int c = blockIdx.x / kTraceCtaStep, r = round - kTraceFirstTile;
    if (blockIdx.x % kTraceCtaStep == 0 && c < kTraceCtas && r >= 0 && r < kTraceTiles) g_trace[c][r][who][event] = clock64();
}
__device__ long long g_trace_cta[kTraceCtas][4];          // kernel entry, set-up done (weights in shared memory, TMEM allocated), last tile done, exit
__device__ __forceinline__ void trace_cta(int event) {
    if (threadIdx.x == 0 && blockIdx.x % kTraceCtaStep == 0 && blockIdx.x / kTraceCtaStep < kTraceCtas) g_trace_cta[blockIdx.x / kTraceCtaStep][event] = clock64();
}
#define TC_TRACE(cond, who, round, event) do { if (cond) trace(who, round, event); } while (0)
#define TC_TRACE_CTA(event) trace_cta(event)
#else
#define TC_TRACE_CTA(event) do { } while (0)
#define TC_TRACE(cond, who, round, event) do { } while (0)
#endif

__device__ __forceinline__ float tanh_mufu(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ uint32_t pack2_f16(float lo, float hi) {
    uint32_t h;
    asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(h) : "f"(hi), "f"(lo));
    return h;
}
__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&v);
}

// this thread's hidden accumulator row (64 columns of TMEM) -> tanh -> fp16 -> its row of the A tile.
// TMEM is read at 64 B per clock per SM (B300_MICROARCH.md): the 32 KB of a tile's hidden accumulator
// take as long to read (512 cycles) as its 8192 tanh take on the four MUFU pipes, so the two must
// overlap: the load of chunk q + 1 is in flight while the tanh of chunk q issue (tcgen05.wait::ld waits
// for every outstanding load, so it is placed after the next load has been issued AND the previous
// chunk's work is done -- by then the load has landed).
// tanh on the FMA pipe: clamp to |x| <= 3.25 and evaluate the odd degree-13 polynomial x P(x^2) (weighted minimax
// fit, tools/fit_tanh_poly.py).  |error| <= 2.0e-3 absolute (1.95e-3 at x = -3.16; P(3.25) = 0.99894 against
// tanh(3.25) = 0.99700) and <= 2.3e-3 relative: that was inside the half-ulp of a bf16 rounding (2^-9 on [0.5, 1)),
// but the fp16 rounding that follows now has a half-ulp of 2^-12 there, so the polynomial columns are about 8 fp16
// half-ulps off -- the dominant term of this kernel's error, an accepted trade (MUFU.TANH is 2^-11 relative).
// tests/test_gpu_policy_numerics.py pins it against a model of this rounding (oracle/policy_oracle.py).
// In this kernel the warps issue no MMAs, so three quarters of
// the issue slots and the whole FMA pipe are idle while the MUFU pipe is the floor: kPolyLanes of every 16 hidden
// activations take this route (the FlashAttention-4 exp2 trick, applied to tanh).
constexpr float kTanhClamp = 3.25f;
__host__ __device__ constexpr float tanh_poly_coef(int k) {    // coefficient of x^(2k+1)
    constexpr float c[7] = {9.977270291e-01f, -3.117916466e-01f, 9.229137325e-02f, -1.838625564e-02f,
                            2.184749761e-03f, -1.380842544e-04f, 3.552717362e-06f};
    return c[k];
}
constexpr int kPolyLanes = 4;         // measured, 2^23 envs: 0: 0.375 ms, 4: 0.344 ms, 6: 0.348 ms, 8: 0.380 ms (warp-MMA kernel: 0.358 ms)
__device__ __forceinline__ float tanh_fma(float x) {
    x = fminf(fmaxf(x, -kTanhClamp), kTanhClamp);
    const float u = x * x;
    float p = tanh_poly_coef(6);
#pragma unroll
    for (int k = 5; k >= 0; --k) p = fmaf(p, u, tanh_poly_coef(k));
    return p * x;
}
// PIPELINED: the load of chunk q + 1 is in flight under the tanh of chunk q (two 16-register buffers); without it
// one buffer, each load awaited before use (16 registers fewer: the fused rollout kernel, which also holds an env).
template <bool PIPELINED>      // the row's 4 chunks of 16 columns
__device__ __forceinline__ void hidden_epilogue(uint32_t taddr_row, __nv_bfloat16* a_tile, int row, int trace_round = 0, int trace_event = 0) {
    constexpr int kChunks = kH / 16;
    uint32_t r[PIPELINED ? 2 : 1][16];
    tmem_ld16(taddr_row, r[0]);
#pragma unroll
    for (int q = 0; q < kChunks; ++q) {
        tmem_wait();                                               // chunk q has landed
        TC_TRACE((threadIdx.x & 31) == 0, (threadIdx.x >> 5) & 3, trace_round, trace_event + 2 * q);
        constexpr int kMask = PIPELINED ? 1 : 0;
        if (PIPELINED && q + 1 < kChunks) tmem_ld16(taddr_row + 16 * (q + 1), r[(q + 1) & kMask]);
        float y[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const float x = __uint_as_float(r[q & kMask][j]);
            // the polynomial lanes are spread over the chunk so that the two pipes interleave
            const bool poly = ((j * kPolyLanes) % 16) < kPolyLanes;
            y[j] = poly ? tanh_fma(x) : tanh_mufu(x);
        }
        if (!PIPELINED && q + 1 < kChunks) tmem_ld16(taddr_row + 16 * (q + 1), r[0]);      // r[0] is dead: lands under the packs and stores
        uint32_t w[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) w[j] = pack2_f16(y[2 * j], y[2 * j + 1]);
        *reinterpret_cast<uint4*>(a_tile + canon(row, 16 * q, kH / 8)) = make_uint4(w[0], w[1], w[2], w[3]);
        *reinterpret_cast<uint4*>(a_tile + canon(row, 16 * q + 8, kH / 8)) = make_uint4(w[4], w[5], w[6], w[7]);
        TC_TRACE((threadIdx.x & 31) == 0, (threadIdx.x >> 5) & 3, trace_round, trace_event + 2 * q + 1);
    }
}

// Weights -> shared memory in the canonical layout, biases split into bf16 hi + lo.  Whole CTA; sync after.
// The global loads are issued in batches of kWBatch per thread before anything is stored: one load per loop trip
// (the first version) made the set-up 23 000 cycles per CTA -- 4 % of a 2^23-env launch -- of exposed L2 latency.
template <int OBS, int ACT>
__device__ __forceinline__ void load_weights(Smem& sm, const float* w1, const float* b1, const float* w2, const float* b2,
                                             const float* w3, const float* b3) {
    const __nv_bfloat16 zero = __float2bfloat16(0.0f);
    auto hi = [](float b) { return __float2bfloat16(b); };
    auto lo = [](float b) { return __float2bfloat16(b - __bfloat162float(__float2bfloat16(b))); };
    // layers 2 and 3: the operand format of the hidden activations (fp16 bit patterns in the same 16-bit tiles)
    auto hid = [](float v) { return __ushort_as_bfloat16(__half_as_ushort(__float2half_rn(v))); };
    auto hid_lo = [](float b) { return __ushort_as_bfloat16(__half_as_ushort(__float2half_rn(b - __half2float(__float2half_rn(b))))); };
    constexpr int kWBatch = 8;
    const int tid = threadIdx.x, nt = blockDim.x;
    for (int base = 0; base < kH * kH; base += kWBatch * nt) {
        float v[kWBatch];
#pragma unroll
        for (int u = 0; u < kWBatch; ++u) { const int e = base + u * nt + tid; v[u] = e < kH * kH ? __ldg(w2 + e) : 0.0f; }
#pragma unroll
        for (int u = 0; u < kWBatch; ++u) { const int e = base + u * nt + tid; if (e < kH * kH) sm.w2[canon(e / kH, e % kH, kH / 8)] = hid(v[u]); }
    }
    float vb1 = 0.0f, vb2 = 0.0f, vb3 = 0.0f;                    // the biases: rows tid of the bias columns / bias tiles
    if (tid < kH) { vb1 = __ldg(b1 + tid); vb2 = __ldg(b2 + tid); }
    if (tid < ACT) vb3 = __ldg(b3 + tid);
    for (int base = 0; base < kH * kK1; base += kWBatch * nt) {
        float v[kWBatch];
#pragma unroll
        for (int u = 0; u < kWBatch; ++u) { const int e = base + u * nt + tid, n = e / kK1, k = e % kK1; v[u] = (e < kH * kK1 && k < OBS) ? __ldg(w1 + n * OBS + k) : 0.0f; }
#pragma unroll
        for (int u = 0; u < kWBatch; ++u) {
            const int e = base + u * nt + tid, n = e / kK1, k = e % kK1;
            if (e < kH * kK1 && k < 14) sm.w1[canon(n, k, kK1 / 8)] = __float2bfloat16(v[u]);          // columns 14, 15: the bias, below
        }
    }
    {
        float v[kWBatch];
        static_assert(kN3 * kH <= kWBatch * 128, "one batch covers layer 3");
#pragma unroll
        for (int u = 0; u < kWBatch; ++u) { const int e = u * nt + tid, n = e / kH; v[u] = (e < kN3 * kH && n < ACT) ? __ldg(w3 + e) : 0.0f; }
#pragma unroll
        for (int u = 0; u < kWBatch; ++u) { const int e = u * nt + tid; if (e < kN3 * kH) sm.w3[canon(e / kH, e % kH, kH / 8)] = hid(v[u]); }
    }
    if (tid < kH) {
        sm.w1[canon(tid, 14, kK1 / 8)] = hi(vb1); sm.w1[canon(tid, 15, kK1 / 8)] = lo(vb1);
#pragma unroll
        for (int k = 0; k < kK1; ++k) sm.b2[canon(tid, k, kK1 / 8)] = k == 0 ? hid(vb2) : (k == 1 ? hid_lo(vb2) : zero);
    }
    if (tid < kN3) {
#pragma unroll
        for (int k = 0; k < kK1; ++k) sm.b3[canon(tid, k, kK1 / 8)] = (tid < ACT && k == 0) ? hid(vb3) : ((tid < ACT && k == 1) ? hid_lo(vb3) : zero);
    }
    for (int e = tid; e < 8 * kK1; e += nt) {
        const int r = e / kK1, k = e % kK1;
        sm.ones[canon(r, k, kK1 / 8)] = k < 2 ? __ushort_as_bfloat16((unsigned short)0x3C00u) : zero;     // 1.0 in the hidden A format (fp16: 0x3C00)
    }
}

struct Args {
    const float* state; int64_t stride, env_stride, n;   // fp32 state: float4 `pl` of env i at pl * stride + i * env_stride
    const float *w1, *b1, *w2, *b2, *w3, *b3;
    float out_scale, out_offset;
    float* action;                                   // [n][ACT]
};

// The MMA warp runs warp-uniformly: every descriptor is built once, outside the elected branch, so the compiler keeps
// them in uniform registers; the elected lane then issues a layer's MMAs and the commit back to back.  (Issued from
// inside an `if (lane == 0)` branch, each MMA was preceded by R2UR moves and descriptor arithmetic: the timeline of
// tools/microbench/policy_tc_trace.cu showed 250 / 570 / 600 cycles to ISSUE layers 1 / 2 / 3 -- 28 % of a tile's
// 5100-cycle chain.)
struct LayerDescs {
    uint64_t a1, w1, a[kH / 16], w2[kH / 16], ones, b2, w3[kH / 16], b3;
    uint32_t d_hidden, d_out;
};
__device__ __forceinline__ LayerDescs make_layer_descs(Smem& sm, uint32_t tmem_base) {
    constexpr uint32_t kLBO = 128, kSBO16 = (kK1 / 8) * 128, kSBO64 = (kH / 8) * 128, kStep = 256;   // one K = 16 step = two chunks
    LayerDescs d;
    SlotSmem& ss = sm.slot;
    d.a1 = make_desc(ss.a1(), kLBO, kSBO16); d.w1 = make_desc(sm.w1, kLBO, kSBO16);
#pragma unroll
    for (int j = 0; j < kH / 16; ++j) {
        d.a[j] = make_desc(reinterpret_cast<const char*>(ss.a) + j * kStep, kLBO, kSBO64);
        d.w2[j] = make_desc(reinterpret_cast<const char*>(sm.w2) + j * kStep, kLBO, kSBO64);
        d.w3[j] = make_desc(reinterpret_cast<const char*>(sm.w3) + j * kStep, kLBO, kSBO64);
    }
    d.ones = make_desc(sm.ones, kLBO, kOnesSBO); d.b2 = make_desc(sm.b2, kLBO, kSBO16); d.b3 = make_desc(sm.b3, kLBO, kSBO16);
    d.d_hidden = tmem_base + kColHidden; d.d_out = tmem_base + kColOut;
    return d;
}
// the MMAs of layer `layer` (1..3), committed to `done`
__device__ __forceinline__ void issue_layer_uniform(const LayerDescs& d, int layer, uint64_t* done) {     // whole warp, converged
    constexpr uint32_t idesc1 = make_idesc(kH), idesc64 = make_idesc(kH, false), idesc16 = make_idesc(kN3, false);
    fence_after_sync();
    if (elect_one()) {
        if (layer == 1) {            // D[128 x 64] = A1[128 x 16] W1^T (bias in columns 14, 15)
            mma_bf16(d.d_hidden, d.a1, d.w1, idesc1, 0u);
        } else if (layer == 2) {     // D[128 x 64] = A[128 x 64] W2^T + ones b2^T
#pragma unroll
            for (int j = 0; j < kH / 16; ++j) mma_bf16(d.d_hidden, d.a[j], d.w2[j], idesc64, j > 0 ? 1u : 0u);
            mma_bf16(d.d_hidden, d.ones, d.b2, idesc64, 1u);
        } else {                     // D[128 x 16] = A[128 x 64] W3^T + ones b3^T
#pragma unroll
            for (int j = 0; j < kH / 16; ++j) mma_bf16(d.d_out, d.a[j], d.w3[j], idesc16, j > 0 ? 1u : 0u);
            mma_bf16(d.d_out, d.ones, d.b3, idesc16, 1u);
        }
        mma_commit(done);
    }
    __syncwarp();
}

// this thread's observation -> its row of the slot's layer-1 A tile (16 bf16: OBS values, zeros, 1, 1)
template <int FIRST, int OBS>
__device__ __forceinline__ void write_obs_row(SlotSmem& ss, int row, const float4 (&p)[3]) {
    const float s[12] = {p[0].x, p[0].y, p[0].z, p[0].w, p[1].x, p[1].y, p[1].z, p[1].w, p[2].x, p[2].y, p[2].z, p[2].w};
    float x[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) x[j] = j < OBS ? s[(FIRST + j) % 12] : ((j == 14 || j == 15) ? 1.0f : 0.0f);
    *reinterpret_cast<uint4*>(ss.a1() + canon(row, 0, kK1 / 8)) = make_uint4(pack2(x[0], x[1]), pack2(x[2], x[3]), pack2(x[4], x[5]), pack2(x[6], x[7]));
    *reinterpret_cast<uint4*>(ss.a1() + canon(row, 8, kK1 / 8)) = make_uint4(pack2(x[8], x[9]), pack2(x[10], x[11]), pack2(x[12], x[13]), pack2(x[14], x[15]));
    fence_async_smem();
}
// the same from the 12 state components a thread holds in registers (the fused rollout kernel)
template <int FIRST, int OBS>
__device__ __forceinline__ void write_obs_row(SlotSmem& ss, int row, const float (&s)[12]) {
    const float4 p[3] = {make_float4(s[0], s[1], s[2], s[3]), make_float4(s[4], s[5], s[6], s[7]), make_float4(s[8], s[9], s[10], s[11])};
    write_obs_row<FIRST, OBS>(ss, row, p);
}

__device__ __forceinline__ void tmem_alloc(Smem& sm) {         // warp 0, converged
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" :: "r"(smem_addr(&sm.tmem_base)), "n"(kTmemCols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_free(uint32_t base) {     // warp 0, converged
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(base), "n"(kTmemCols) : "memory");
}

constexpr int kCtasPerSm = 7;                       // x kTmemCols <= the SM's 512 TMEM columns
// Tile k + 1 of a CTA (tile 0 is blockIdx.x): the answer to try_cancel k, read by every thread of both roles from
// clc_resp[k & 1] once clc_bar[k & 1] has completed.
__device__ __forceinline__ uint32_t next_tile(Smem& sm, int k, uint32_t& clc_phase) {
    bar_wait(&sm.clc_bar[k & 1], (clc_phase >> (k & 1)) & 1u); clc_phase ^= 1u << (k & 1);
    return clc_response(&sm.clc_resp[k & 1]);
}
// the MMA warp (converged): ask for the tile after next -- answer k + 1 -- unless answer k was "nothing left"
__device__ __forceinline__ void request_tile(Smem& sm, int k_next) {
    if (elect_one()) { fence_async_smem(); clc_try_cancel(&sm.clc_resp[k_next & 1], &sm.clc_bar[k_next & 1]); }
    __syncwarp();
}
constexpr int kThreads = kTile + 32;      // the epilogue warps + the MMA warp

// ---- where a tile's observation rows come from (the source) and where its outputs go (the head) ----
// Sources and heads are types only: they read their pointers and sizes from the kernel's __grid_constant__ arguments
// in place (copied into a struct, the policy kernel's values stayed in registers and spilled).  A source also says
// which rows are evaluated: selected(i) for one row and, where kSelect, tile_live(tile) for the whole tile (called by
// every warp of both roles, converged; each reaches the same answer from the same bytes, with no message between them).
// The env state (Args): float4 `pl` of env i at pl * stride + i * env_stride; the observation is components
// FIRST .. FIRST + OBS - 1.
template <int FIRST_, int OBS_>
struct StateRows {
    static constexpr int FIRST = FIRST_, OBS = OBS_;
    static constexpr bool kSelect = false;
    template <class A> __device__ static __forceinline__ void fetch(const A& a, int64_t i, float4 (&p)[3]) {
        const float4* env = reinterpret_cast<const float4*>(a.state) + i * a.env_stride;
        p[0] = env[0]; p[1] = env[a.stride]; p[2] = env[2 * a.stride];
    }
    template <class A> __device__ static __forceinline__ bool selected(const A&, int64_t) { return true; }
    template <class A> __device__ static __forceinline__ bool tile_live(const A&, uint32_t) { return true; }
};
// Packed fp32 observation rows (ValueArgs): row r at rows + r * row_stride floats (row_stride >= OBS; 4-byte alignment
// is enough: the loads are scalar, and they are not the bound).  With `select`, only rows with select[r] & mask are
// evaluated; a tile without one skips its MMAs and epilogue.
template <int OBS_>
struct ObsRows {
    static constexpr int FIRST = 0, OBS = OBS_;
    static constexpr bool kSelect = true;
    template <class A> __device__ static __forceinline__ void fetch(const A& a, int64_t i, float4 (&p)[3]) {
        float s[12];
#pragma unroll
        for (int j = 0; j < 12; ++j) s[j] = j < OBS ? __ldg(a.rows + i * a.row_stride + j) : 0.0f;
        p[0] = make_float4(s[0], s[1], s[2], s[3]); p[1] = make_float4(s[4], s[5], s[6], s[7]); p[2] = make_float4(s[8], s[9], s[10], s[11]);
    }
    template <class A> __device__ static __forceinline__ bool selected(const A& a, int64_t i) {
        return !a.select || (__ldg(a.select + i) & a.select_mask) != 0;
    }
    template <class A> __device__ static __forceinline__ bool tile_live(const A& a, uint32_t tile) {   // the tile's 128 select bytes, 4 per lane
        if (!a.select) return true;
        bool any = false;
#pragma unroll
        for (int q = 0; q < kTile / 32; ++q) {
            const int64_t i = (int64_t)tile * kTile + q * 32 + (threadIdx.x & 31);
            any |= i < a.n && (__ldg(a.select + i) & a.select_mask) != 0;
        }
        return __any_sync(0xffffffffu, any);
    }
};
// the policy's action rows [n][ACT] (Args): out_offset + out_scale * tanh(layer 3)
template <int ACT_>
struct ActionHead {
    static constexpr int ACT = ACT_;
    template <class A> __device__ static __forceinline__ void store(const A& a, int64_t i, const float (&pre)[4]) {
        float act[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) act[j] = fmaf(a.out_scale, tanh_mufu(pre[j]), a.out_offset);
        if constexpr (ACT == 4) reinterpret_cast<float4*>(a.action)[i] = make_float4(act[0], act[1], act[2], act[3]);
        else if constexpr (ACT == 2) reinterpret_cast<float2*>(a.action)[i] = make_float2(act[0], act[1]);
        else a.action[i] = act[0];
    }
};
// the critic's value [n] (ValueArgs): layer 3's accumulator column 0, no tanh
struct ValueHead {
    static constexpr int ACT = 1;
    template <class A> __device__ static __forceinline__ void store(const A& a, int64_t i, const float (&pre)[4]) { a.value[i] = pre[0]; }
};

// observation rows -> outputs.  Persistent, warp-specialised CTAs (weights converted once per CTA), 128 rows
// per tile, one tile in flight per CTA, the tiles taken by cluster launch control (next_tile).
//   epilogue warps   one thread per env row: pull the accumulator out of TMEM, tanh, fp16, write it to shared
//              memory as the next layer's A operand, arrive on ready; after layer 3 store the env's action and
//              put the NEXT tile's observation row in place.  They never wait for one another: the only thing
//              a thread waits for is done of the layer it is about to read.
//   last warp  warp-uniform, one elected lane issuing: waits for ready (all epilogue threads), issues the
//              layer's tcgen05.mma, commits them to done.
// The MUFU pipe is the floor (132 tanh per env) and what keeps it busy is WARPS: every wait in an epilogue
// warp (mbarrier, TMEM load, shared-memory fence) has to be covered by another warp's tanh.
// History, 2^23 envs (warp-MMA kernel of copter_policy.cuh: 0.358 ms, XU 72 %):
//   one tile per CTA, __syncthreads + thread 0 issuing, 4 CTAs/SM          0.627 ms  (CTAs march in step)
//   two tiles in flight per CTA, still __syncthreads, 2 CTAs/SM            0.484 ms
//   + MMA warp and mbarriers instead of __syncthreads                      0.428 ms  (XU 60 %; three tiles: 0.437)
//   one tile in flight, 4 CTAs/SM (16 epilogue warps per SM instead of 8)  0.374 ms
//   two threads per row: 3 CTAs/SM (24 epilogue warps) 0.406 ms, 4 CTAs/SM (32 warps, 56 registers) 0.387 ms: more warps do not help
//   one tile in flight, 4 CTAs/SM, 4 of every 16 hidden tanh on the FMA pipe 0.344 ms  (profiles/r2_policy_kernels_*)
//   64 TMEM columns per tile (layer 3's output reuses the hidden columns), layer-1 A tile aliased into the hidden
//   A tile (34.5 KB of shared memory per CTA): 5 CTAs/SM 0.321 ms  <- shipped; 6 CTAs/SM (64 registers) 0.322 ms;
//   6 of 16 tanh as polynomials 0.330, 8 of 16 0.355 (profiles/r2_sweep_policy_tc_ctas.txt)
//   (tools/microbench/tmem_rates.cu, profiles/r2_tmem_rates.txt: TMEM read-back is NOT the floor -- 184 B/clk/SM from
//   one CTA, 370 B/clk/SM from four, and tcgen05.ld overlaps tanh.approx completely; the MUFU floor is 0.19 ms)
// (The loop with several tiles in flight per CTA or two epilogue threads per row: the last tree that has it is
// commit d11af01.)
// A tile without a selected row (tile_live false, ObsRows only) costs one handshake instead of three layers: the
// epilogue threads arrive on ready once (the next tile's rows), the MMA warp waits for it, issues nothing and arrives on
// done once, and the epilogue threads wait for that before they read the next tile's answer -- without that wait they
// could complete two phases of ready before the MMA warp has seen the first.
template <class Src, class Head, class A>
__device__ __forceinline__ void mlp_tc_tiles(const A& a) {
    constexpr int FIRST = Src::FIRST, OBS = Src::OBS, ACT = Head::ACT;
    static_assert(OBS <= 12 && ACT <= 4, "tile shapes");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw);
    const int t = threadIdx.x, warp = t >> 5;
    constexpr int kMmaWarp = kTile / 32;
    TC_TRACE_CTA(0);
    if (t == 0) {
        bar_init(&sm.done, 1); bar_init(&sm.ready, kTile);
        bar_init(&sm.clc_bar[0], 1); bar_init(&sm.clc_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kMmaWarp) tmem_alloc(sm);
    load_weights<OBS, ACT>(sm, a.w1, a.b1, a.w2, a.b2, a.w3, a.b3);
    fence_async_smem();
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    TC_TRACE_CTA(1);
    const uint32_t tmem_base = sm.tmem_base;
    auto tile_live = [&](uint32_t tl) {          // whole warp, converged
        if constexpr (Src::kSelect) return tl != kNoTile && Src::tile_live(a, tl);
        else return true;
    };

    // Tile k of this CTA: k = 0 is blockIdx.x; tile k + 1 is the answer to try_cancel k.
    // The MMA warp keeps one try_cancel in flight; both roles read answer k from clc_resp[k & 1] after clc_bar[k & 1]
    // -- the epilogue threads after they have handed layer 2 its A tile, i.e. while they would only wait -- and
    // clc_resp[k & 1] is re-armed (try_cancel k + 2) only after every epilogue thread has arrived for layer 1 of tile
    // k + 1, which it does after that read.
    if (warp == kMmaWarp) {
        const LayerDescs d = make_layer_descs(sm, tmem_base);
        uint32_t tile = blockIdx.x, phase = 0, clc_phase = 0;
        bool live = tile_live(tile);
        request_tile(sm, 0);
        for (int k = 0; tile != kNoTile; ++k) {
            bar_wait(&sm.ready, phase); phase ^= 1u;
            TC_TRACE((t & 31) == 0, 4, k, 0);
            if (live) issue_layer_uniform(d, 1, &sm.done);
            else { if (elect_one()) bar_arrive(&sm.done); __syncwarp(); }
            TC_TRACE((t & 31) == 0, 4, k, 2);
            const uint32_t nxt = next_tile(sm, k, clc_phase);
            if (nxt != kNoTile) request_tile(sm, k + 1);          // (a failed try_cancel is the last one)
            if (live) {
#pragma unroll
                for (int layer = 2; layer <= 3; ++layer) {
                    bar_wait(&sm.ready, phase); phase ^= 1u;
                    TC_TRACE((t & 31) == 0, 4, k, 3 * (layer - 1));
                    issue_layer_uniform(d, layer, &sm.done);
                    TC_TRACE((t & 31) == 0, 4, k, 3 * (layer - 1) + 2);
                }
            }
            tile = nxt;
            live = tile_live(tile);
        }
    } else {
        const int row = t;
        const uint32_t lane_base = tmem_base + ((uint32_t)(warp * 32) << 16);       // this warp's quarter of the 128 TMEM lanes
        auto fetch = [&](uint32_t tl, bool tl_live, float4 (&p)[3]) {
            const int64_t i = (int64_t)tl * kTile + row;
            if (tl != kNoTile && tl_live && i < a.n) Src::fetch(a, i, p);
            else p[0] = p[1] = p[2] = make_float4(0.f, 0.f, 0.f, 0.f);
        };
        uint32_t tile = blockIdx.x, phase = 0, clc_phase = 0;
        bool live = tile_live(tile);
        float4 nxt[3];
        fetch(tile, live, nxt);
        write_obs_row<FIRST, OBS>(sm.slot, row, nxt);
        fence_before_sync();
        bar_arrive(&sm.ready);
        for (int k = 0; tile != kNoTile; ++k) {
            uint32_t nxt_tile = kNoTile;
            bool nxt_live = false;
            float pre[4];
            if (live) {
#pragma unroll
                for (int layer = 1; layer <= 2; ++layer) {
                    bar_wait(&sm.done, phase); phase ^= 1u;
                    fence_after_sync();
                    TC_TRACE((t & 31) == 0, warp, k, 3 * (layer - 1));
                    hidden_epilogue<true>(lane_base + kColHidden, sm.slot.a, row, k, 12 + 8 * (layer - 1));      // (layer 2 overwrites the tile its finished MMAs read)
                    TC_TRACE((t & 31) == 0, warp, k, 3 * (layer - 1) + 1);
                    fence_async_smem();
                    fence_before_sync();
                    bar_arrive(&sm.ready);
                    TC_TRACE((t & 31) == 0, warp, k, 3 * (layer - 1) + 2);
                    if (layer == 1) {                                    // under layer 2's MMAs: which tile is next, and its state on the way
                        nxt_tile = next_tile(sm, k, clc_phase);
                        nxt_live = tile_live(nxt_tile);
                        fetch(nxt_tile, nxt_live, nxt);
                    }
                }
                bar_wait(&sm.done, phase); phase ^= 1u;
                fence_after_sync();
                TC_TRACE((t & 31) == 0, warp, k, 6);
                tmem_ld4(lane_base + kColOut, pre);
                TC_TRACE((t & 31) == 0, warp, k, 7);
            } else {                                                 // the MMA warp has taken this tile's handshake
                bar_wait(&sm.done, phase); phase ^= 1u;
                nxt_tile = next_tile(sm, k, clc_phase);
                nxt_live = tile_live(nxt_tile);
                fetch(nxt_tile, nxt_live, nxt);
            }
            if (nxt_tile != kNoTile) {                               // the next tile's observation row first: the MMA warp is waiting for it
                write_obs_row<FIRST, OBS>(sm.slot, row, nxt);
                fence_before_sync();
                bar_arrive(&sm.ready);
                TC_TRACE((t & 31) == 0, warp, k, 8);
            }
            const int64_t i = (int64_t)tile * kTile + row;
            if (live && i < a.n && Src::selected(a, i)) Head::store(a, i, pre);
            tile = nxt_tile;
            live = nxt_live;
        }
    }
    TC_TRACE_CTA(2);
    fence_before_sync();
    __syncthreads();
    if (warp == kMmaWarp) tmem_free(tmem_base);
    TC_TRACE_CTA(3);
}

// env state -> action rows (copter_policy_mlp_strided_f32)
template <int FIRST, int OBS, int ACT>
__global__ void __launch_bounds__(kThreads, kCtasPerSm)
copter_mlp_policy_tc_kernel(const __grid_constant__ Args a) {
    mlp_tc_tiles<StateRows<FIRST, OBS>, ActionHead<ACT>>(a);
}

// observation rows -> values (copter_value_mlp_f32): the critic O -> 64 -> 64 -> 1, layer 3 linear
struct ValueArgs {
    const float* rows; int64_t row_stride, n;
    const uint8_t* select; uint32_t select_mask;     // select nullable
    const float *w1, *b1, *w2, *b2, *w3, *b3;        // w3 [1][64], b3 [1]
    float* value;                                    // [n]
};
// 5 CTAs per SM, 80 registers (__maxnreg__): the selection adds state to every role, and at the policy's 7 CTAs (56 registers) or at
// 6 (64) the kernel spilled 8-52 bytes per thread; unbounded it takes 72-80.  The policy kernel measured 0.321 ms at 5
// CTAs per SM and 0.322 at 6 (profiles/r2_sweep_policy_tc_ctas.txt).
constexpr int kValueCtasPerSm = 5;
template <int OBS>
__global__ void __maxnreg__(65536 / (kThreads * kValueCtasPerSm) / 8 * 8)
copter_value_tc_kernel(const __grid_constant__ ValueArgs a) {
    mlp_tc_tiles<ObsRows<OBS>, ValueHead>(a);
}

}  // namespace tc
}  // namespace copter
