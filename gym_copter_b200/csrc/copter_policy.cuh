// copter_policy.cuh -- the small tanh MLP policy of BASELINE.json configs[4] (O -> 64 -> 64 -> A,
// SURVEY.md 8d "config 5") evaluated by a warp for its 32 envs straight from the fp32 state each
// lane holds in registers.  Two kernels use it (copter_kernels.cu): copter_mlp_policy_kernel
// (env state -> action rows, for policy-in-the-loop rollouts that step with copter_step_*)
// and copter_policy_rollout_kernel (policy + env step for T steps in ONE launch, the state
// never leaving registers).  In PyTorch this policy costs 4.2 ms per step for 2^23 envs (three
// GEMMs with [N,64] intermediates through HBM plus separate tanh passes) against 0.21 ms for
// the env step itself.
//
// One warp = 32 envs = two 16-row tiles of warp-level tensor-core MMAs (mma.sync.m16n8k16,
// bf16 inputs, fp32 accumulation).  The accumulator fragment of layer L is exactly the
// A-operand fragment of layer L+1 (n-tiles 2k, 2k+1 -> k-tile k), so between layers there is
// only tanh (MUFU.TANH) + bf16 packing, all in registers; the bias enters as the accumulator's
// initial value, and layer 3 consumes each pair of layer-2 n-tiles as soon as it exists, so the
// second hidden activation is never held whole.  Both row tiles share every weight fragment
// load.  The kernel is bound by the MUFU (XU) pipe -- 132 tanh per env -- which is why the
// warp-level MMA is enough here: tcgen05/TMEM would not move the XU floor.
// Weights live in shared memory as bf16 in FRAGMENT ORDER (the 64-/128-bit word a lane needs
// for an MMA sits at [tile][lane]), so B operands arrive as conflict-free LDS.64 / LDS.128.
#pragma once

#include <cuda_bf16.h>

namespace copter {

constexpr int kPolH = 64;            // hidden width
constexpr int kPolIn = 16;           // observation padded to one k-tile
constexpr int kPolOut = 8;           // actions padded to one n-tile
constexpr int kPolXStride = kPolIn + 8;   // bf16 elements per env row of the input tile (48 B: ldmatrix rows hit distinct banks)

// torch.nn.Linear layouts: W[out][in], b[out], fp32 device memory
struct PolicyWeights {
    const float *w1, *b1, *w2, *b2, *w3, *b3;
    float out_scale, out_offset;     // action = out_offset + out_scale * tanh(.)
};

struct PolicySmem {
    uint2 w1[8][32];                 // layer 1: [n-tile][lane] -> {b0, b1} of the single k-tile
    uint4 w2[8][2][32];              // layer 2: [n-tile][k-tile pair][lane] -> {b0, b1 of k-tile 2p, b0, b1 of k-tile 2p+1}
    uint4 w3[2][32];                 // layer 3: [k-tile pair][lane]
    float4 b1[8][4], b2[8][4], b3[4];   // [n-tile][t] -> bias of columns 2t, 2t+1, twice: an accumulator quad as loaded
};
// per-warp scratch: the bf16 input rows (ldmatrix source) and the fp32 pre-activation action rows
struct PolicyWarpTile {
    __nv_bfloat16 x[32 * kPolXStride];
    float act[32 * 4];
};

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ float tanh_fast(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// hidden activations: two fp32 MUFU.TANH, then one bf16 pair.  (tanh.approx.bf16x2 on the pair rounded to bf16 first is
// not faster on B200 -- measured 0.435 ms vs 0.412 ms for 2^23 envs: the packed form costs two XU slots -- and is less
// accurate; an FMA-pipe polynomial for some of the n-tiles gained 2 % at 1/8 of them and lost beyond
// (profiles/r1_sweep_policy_poly_tanh.txt).  Both knobs are removed; the last tree that has them is commit d11af01.)
__device__ __forceinline__ uint32_t tanh_pack(float lo, float hi) {
    return pack_bf16(tanh_fast(lo), tanh_fast(hi));
}
// D = A B + D
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
// D = A B + C with C = the bias quad (x, y, x, y: the lane's two columns for both row halves) exactly
// as one LDS.128 delivers it, so no register is moved to build the accumulator
__device__ __forceinline__ void mma_bf16_bias(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1, const float4& c) {
    asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%11,%12,%13};"
        : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1), "f"(c.x), "f"(c.y), "f"(c.z), "f"(c.w));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], const void* smem_row) {
    const uint32_t addr = (uint32_t)__cvta_generic_to_shared(smem_row);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}

// Weights -> shared memory: bf16, zero-padded to the tile shapes, in mma.m16n8k16 B-fragment
// order.  For the lane (g = lane / 4, t = lane % 4), n-tile nt and k-tile kt the fragment is
//   b0 = W[8 nt + g][16 kt + 2t, +1],  b1 = W[8 nt + g][16 kt + 8 + 2t, +1]      (B[k][n] = W[n][k]).
// Call with the whole CTA, then __syncthreads().
template <int OBS, int ACT>
__device__ __forceinline__ void policy_load_weights(PolicySmem& sm, const PolicyWeights& w) {
    const auto w1 = [&](int n, int k) { return k < OBS ? w.w1[n * OBS + k] : 0.0f; };
    const auto w2 = [&](int n, int k) { return w.w2[n * kPolH + k]; };
    const auto w3 = [&](int n, int k) { return n < ACT ? w.w3[n * kPolH + k] : 0.0f; };
    for (int e = threadIdx.x; e < 8 * 32; e += blockDim.x) {
        const int nt = e >> 5, lane = e & 31, n = 8 * nt + (lane >> 2), k = 2 * (lane & 3);
        sm.w1[nt][lane] = make_uint2(pack_bf16(w1(n, k), w1(n, k + 1)), pack_bf16(w1(n, k + 8), w1(n, k + 9)));
    }
    for (int e = threadIdx.x; e < 8 * 2 * 32; e += blockDim.x) {
        const int nt = e >> 6, kp = (e >> 5) & 1, lane = e & 31, n = 8 * nt + (lane >> 2), k = 32 * kp + 2 * (lane & 3);
        sm.w2[nt][kp][lane] = make_uint4(pack_bf16(w2(n, k), w2(n, k + 1)), pack_bf16(w2(n, k + 8), w2(n, k + 9)),
                                         pack_bf16(w2(n, k + 16), w2(n, k + 17)), pack_bf16(w2(n, k + 24), w2(n, k + 25)));
    }
    for (int e = threadIdx.x; e < 2 * 32; e += blockDim.x) {
        const int kp = e >> 5, lane = e & 31, n = lane >> 2, k = 32 * kp + 2 * (lane & 3);
        sm.w3[kp][lane] = make_uint4(pack_bf16(w3(n, k), w3(n, k + 1)), pack_bf16(w3(n, k + 8), w3(n, k + 9)),
                                     pack_bf16(w3(n, k + 16), w3(n, k + 17)), pack_bf16(w3(n, k + 24), w3(n, k + 25)));
    }
    for (int e = threadIdx.x; e < 8 * 4; e += blockDim.x) {
        const int c = 8 * (e >> 2) + 2 * (e & 3);
        sm.b1[e >> 2][e & 3] = make_float4(w.b1[c], w.b1[c + 1], w.b1[c], w.b1[c + 1]);
        sm.b2[e >> 2][e & 3] = make_float4(w.b2[c], w.b2[c + 1], w.b2[c], w.b2[c + 1]);
    }
    if (threadIdx.x < 4) {
        const int c = 2 * threadIdx.x;
        const float x = c < ACT ? w.b3[c] : 0.0f, y = c + 1 < ACT ? w.b3[c + 1] : 0.0f;
        sm.b3[threadIdx.x] = make_float4(x, y, x, y);
    }
}

// The policy for the 32 envs of a warp.  `s` is this lane's env state (zeros for a lane without
// an env); the observation is components FIRST .. FIRST+OBS-1.  Returns the lane's action row
// (before the env's clip).  Warp-uniform call: every lane must take part.
template <int FIRST, int OBS, int ACT>
__device__ __forceinline__ void policy_forward_warp(const PolicySmem& sm, PolicyWarpTile& wt, int lane, const float (&s)[12],
                                                    float out_scale, float out_offset, float (&action)[ACT]) {
    static_assert(OBS <= kPolIn && ACT <= 4 && FIRST + OBS <= 12, "policy tile shapes");
    const int g = lane >> 2, t = lane & 3;

    // this lane's observation -> 16 bf16 inputs (zero padded) -> the warp's input tile
    uint32_t xin[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float lo = (2 * j < OBS) ? s[(FIRST + 2 * j) % 12] : 0.0f;
        const float hi = (2 * j + 1 < OBS) ? s[(FIRST + 2 * j + 1) % 12] : 0.0f;
        xin[j] = pack_bf16(lo, hi);
    }
    uint4* xrow = reinterpret_cast<uint4*>(wt.x + lane * kPolXStride);
    xrow[0] = make_uint4(xin[0], xin[1], xin[2], xin[3]);
    xrow[1] = make_uint4(xin[4], xin[5], xin[6], xin[7]);
    __syncwarp();

    // both row tiles of 16 envs are carried through the layers together: every weight fragment load serves
    // both tiles and the two accumulator chains interleave (one tile at a time: half the live registers, twice
    // the fragment loads -- slower, profiles/r1_sweep_policy_occupancy.txt)
    constexpr int MT = 2;
    // layer-1 A fragments: four 8x8 matrices per row tile (rows 0-7 / 8-15 x k 0-7 / 8-15)
    uint32_t a1[MT][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
        const int j = lane >> 3, r = lane & 7;
        ldmatrix_x4(a1[mt], wt.x + (16 * mt + 8 * (j & 1) + r) * kPolXStride + 8 * (j >> 1));
    }

    // ---- layer 1: [16 MT x 16] x [16 x 64], activations kept as the A fragments of layer 2 ----
    uint32_t h[MT][4][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
        const uint2 b = sm.w1[nt][lane];
        const float4 bias = sm.b1[nt][t];
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            float c[4];
            mma_bf16_bias(c, a1[mt], b.x, b.y, bias);
            h[mt][nt >> 1][(nt & 1) * 2 + 0] = tanh_pack(c[0], c[1]);      // rows g
            h[mt][nt >> 1][(nt & 1) * 2 + 1] = tanh_pack(c[2], c[3]);      // rows g + 8
        }
    }

    // ---- layer 2: [16 MT x 64] x [64 x 64], two n-tiles at a time, each pair feeding one k-tile of
    // ---- layer 3: [16 MT x 64] x [64 x 8]
    float c3[MT][4];
#pragma unroll
    for (int kt3 = 0; kt3 < 4; ++kt3) {
        uint32_t a3[MT][4];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int nt = 2 * kt3 + half;
            const float4 bias = sm.b2[nt][t];
            float c[MT][4];
#pragma unroll
            for (int kp = 0; kp < 2; ++kp) {
                const uint4 b = sm.w2[nt][kp][lane];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    if (kp == 0) mma_bf16_bias(c[mt], h[mt][0], b.x, b.y, bias);
                    else         mma_bf16(c[mt], h[mt][2], b.x, b.y);
                    mma_bf16(c[mt], h[mt][2 * kp + 1], b.z, b.w);
                }
            }
#pragma unroll
            for (int mt = 0; mt < MT; ++mt) {
                a3[mt][half * 2 + 0] = tanh_pack(c[mt][0], c[mt][1]);
                a3[mt][half * 2 + 1] = tanh_pack(c[mt][2], c[mt][3]);
            }
        }
        const uint4 b = sm.w3[kt3 >> 1][lane];
        const uint32_t b0 = (kt3 & 1) ? b.z : b.x, b1 = (kt3 & 1) ? b.w : b.y;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            if (kt3 == 0) mma_bf16_bias(c3[mt], a3[mt], b0, b1, sm.b3[t]);
            else          mma_bf16(c3[mt], a3[mt], b0, b1);
        }
    }

    // lanes t < 2 hold columns 2t, 2t+1 (< 4) of rows g and g + 8 of each row tile: hand every
    // env's pre-activation row back to its own lane, which applies the output tanh once
    if (t < 2) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
            *reinterpret_cast<float2*>(wt.act + (16 * mt + g) * 4 + 2 * t) = make_float2(c3[mt][0], c3[mt][1]);
            *reinterpret_cast<float2*>(wt.act + (16 * mt + g + 8) * 4 + 2 * t) = make_float2(c3[mt][2], c3[mt][3]);
        }
    }
    __syncwarp();
    const float4 pre = *reinterpret_cast<const float4*>(wt.act + lane * 4);
    const float p[4] = {pre.x, pre.y, pre.z, pre.w};
#pragma unroll
    for (int j = 0; j < ACT; ++j) action[j] = fmaf(out_scale, tanh_fast(p[j]), out_offset);
    __syncwarp();
}

struct PolicyArgs {
    const float* state; int64_t stride, env_stride, n;   // fp32 state: float4 `pl` of env i at pl * stride + i * env_stride
    PolicyWeights w;
    float* action;                                   // [n][act]
};

constexpr int kPolicyCtasPerSm = 5;      // measured (profiles/r1_sweep_policy_occupancy.txt, 2^23 envs): 3: 0.386, 4: 0.373, 5: 0.359, 6: 0.368 ms

// env state -> action rows.  Persistent CTAs: the weights are converted once per CTA.
template <int FIRST, int OBS, int ACT>
__global__ void __launch_bounds__(128, kPolicyCtasPerSm)
copter_mlp_policy_kernel(const __grid_constant__ PolicyArgs a) {
    __shared__ __align__(16) PolicySmem sm;
    __shared__ __align__(16) PolicyWarpTile wtile[4];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    policy_load_weights<OBS, ACT>(sm, a.w);
    __syncthreads();

    const int64_t n_warp_tiles = (a.n + 31) / 32;
    for (int64_t wt = (int64_t)blockIdx.x * 4 + warp; wt < n_warp_tiles; wt += (int64_t)gridDim.x * 4) {
        const int64_t i = wt * 32 + lane;
        float s[12];
        if (i < a.n) {
            // (env_stride made opaque inside the loop: otherwise the compiler carries i * env_stride as one more 64-bit
            // induction variable across the network, and this 96-register kernel spills 136 instead of 56 bytes)
            int64_t env_stride = a.env_stride;
            asm volatile("" : "+l"(env_stride));
            const float4* env = reinterpret_cast<const float4*>(a.state) + i * env_stride;
#pragma unroll
            for (int pl = 0; pl < 3; ++pl) {
                const float4 v = env[(int64_t)pl * a.stride];
                s[4 * pl] = v.x; s[4 * pl + 1] = v.y; s[4 * pl + 2] = v.z; s[4 * pl + 3] = v.w;
            }
        } else {
#pragma unroll
            for (int j = 0; j < 12; ++j) s[j] = 0.0f;
        }
        float act[ACT];
        policy_forward_warp<FIRST, OBS, ACT>(sm, wtile[warp], lane, s, a.w.out_scale, a.w.out_offset, act);
        if (i < a.n) {
            if constexpr (ACT == 4) reinterpret_cast<float4*>(a.action)[i] = make_float4(act[0], act[1], act[2], act[3]);
            else if constexpr (ACT == 2) reinterpret_cast<float2*>(a.action)[i] = make_float2(act[0], act[1]);
            else a.action[i] = act[0];
        }
    }
}

}  // namespace copter
