// k1_traffic.cu -- the HBM ceiling of the fp32 K = 1 step's byte pattern, with no physics.
//
// 2^24 envs in the headline's buffers and layout: each env reads its 48-byte state row, its 4-byte meta word
// and its 16-byte action row, and writes the row, the meta word, a 4-byte reward and a 1-byte done flag --
// 125 B per env, what copter_step_kernel<float, LANDER3D> moves at K = 1.  Two access patterns:
//   (a) one CTA per 128-env tile, one thread per env, three 128-bit row loads at a 48-byte stride: the
//       loads of copter_step_kernel;
//   (b) resident CTAs taking tiles from cluster launch control, each tile's inputs brought into a D-stage
//       shared-memory ring by cp.async.bulk (one copy of the rows, one of the actions, one of the meta words),
//       D - 1 tiles ahead of the one being consumed: the loads of copter_step1_kernel.  Swept over D and
//       the CTAs per SM (set through the dynamic shared memory each CTA reserves).
// Stores are plain per-thread stores in both.  Times: CUDA events over 200 back-to-back launches after 20 of
// warm-up, median of 5 such regions; the working set (2.1 GB) is far above L2.
//
// build: nvcc -std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -o tools/microbench/k1_traffic tools/microbench/k1_traffic.cu
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <algorithm>
#include <vector>

#include "../../gym_copter_b200/csrc/copter_policy_tc.cuh"

using namespace copter;

#define CHECK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)

constexpr int kBlock = 128;
constexpr int64_t kEnvs = 1 << 24;

struct Bufs { float4* state; uint32_t* meta; const float4* action; float* reward; uint8_t* done; int64_t n; };

// the per-env "work": enough to keep every loaded word live, nothing more
__device__ __forceinline__ void finish(const Bufs& b, int64_t i, float4 r0, float4 r1, float4 r2, uint32_t m, float4 act) {
    r0.x += act.x; r1.y += act.y; r2.z += act.z; r2.w += act.w;
    b.state[3 * i] = r0; b.state[3 * i + 1] = r1; b.state[3 * i + 2] = r2;
    b.meta[i] = m + 4u;
    b.reward[i] = r0.y + r1.x + r2.x;
    b.done[i] = (uint8_t)(m & 1u);
}

__global__ void __launch_bounds__(kBlock) traffic_direct(const Bufs b) {
    const int64_t i = (int64_t)blockIdx.x * kBlock + threadIdx.x;
    if (i >= b.n) return;
    const float4 r0 = b.state[3 * i], r1 = b.state[3 * i + 1], r2 = b.state[3 * i + 2];
    finish(b, i, r0, r1, r2, b.meta[i], b.action[i]);
}

struct alignas(128) Stage { float4 state[3 * kBlock]; float4 act[kBlock]; uint32_t meta[kBlock]; };

__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(tc::smem_addr(dst)), "l"(src), "r"(bytes), "r"(tc::smem_addr(bar)) : "memory");
}

template <int D>
__global__ void __launch_bounds__(kBlock) traffic_bulk(const Bufs b) {
    __shared__ Stage stage[D];
    __shared__ __align__(8) uint64_t full[D], empty[D], clc_bar;
    __shared__ __align__(16) uint4 clc_resp;
    __shared__ uint32_t tile_of[D], next, clc_phase, fill;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < D; ++s) { tc::bar_init(&full[s], 1); tc::bar_init(&empty[s], kBlock / 32); }
        tc::bar_init(&clc_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        next = blockIdx.x; clc_phase = 0; fill = 0;
    }
    __syncthreads();
    auto produce = [&]() {
        const uint32_t f = fill;
        const int s = f % D;
        if (f >= D) tc::bar_wait(&empty[s], (f / D - 1) & 1u);
        if (tc::elect_one()) {
            const uint32_t t = next;
            tile_of[s] = t;
            if (t != tc::kNoTile) {     // 2^24 envs: every tile is full
                const int64_t row0 = (int64_t)t * kBlock;
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(tc::smem_addr(&full[s])), "r"((uint32_t)sizeof(Stage)) : "memory");
                bulk_load(stage[s].state, b.state + 3 * row0, sizeof(stage[s].state), &full[s]);
                bulk_load(stage[s].act, b.action + row0, sizeof(stage[s].act), &full[s]);
                bulk_load(stage[s].meta, b.meta + row0, sizeof(stage[s].meta), &full[s]);
            } else {
                tc::bar_arrive(&full[s]);
            }
            fill = f + 1;
        }
        __syncwarp();
    };
    if (warp == 0) {
        if (tc::elect_one()) tc::clc_try_cancel(&clc_resp, &clc_bar);
        __syncwarp();
        produce();
    }
    for (uint32_t j = 0;; ++j) {
        if (warp == 0) {
            while (next != tc::kNoTile && fill < j + D) {
                tc::bar_wait(&clc_bar, clc_phase);
                const uint32_t t = tc::clc_response(&clc_resp);
                __syncwarp();
                if (tc::elect_one()) {
                    next = t; clc_phase ^= 1u;
                    if (t != tc::kNoTile) { tc::fence_async_smem(); tc::clc_try_cancel(&clc_resp, &clc_bar); }
                }
                __syncwarp();
                produce();
            }
        }
        const int s = j % D;
        tc::bar_wait(&full[s], (j / D) & 1u);
        const uint32_t tile = tile_of[s];
        if (tile == tc::kNoTile) break;
        const float4* src = stage[s].state + 3 * threadIdx.x;
        const float4 r0 = src[0], r1 = src[1], r2 = src[2], act = stage[s].act[threadIdx.x];
        const uint32_t m = stage[s].meta[threadIdx.x];
        __syncwarp();
        if (lane == 0) tc::bar_arrive(&empty[s]);
        finish(b, (int64_t)tile * kBlock + threadIdx.x, r0, r1, r2, m, act);
    }
}

template <typename Launch>
float time_ms(Launch launch) {
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int w = 0; w < 20; ++w) launch();
    std::vector<float> reps;
    for (int r = 0; r < 5; ++r) {
        cudaEventRecord(e0);
        for (int s = 0; s < 200; ++s) launch();
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
        reps.push_back(ms / 200);
    }
    std::sort(reps.begin(), reps.end());
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return reps[2];
}

template <int D>
int run_bulk(const Bufs& b, int grid, int ctas) {
    // occupancy set through the dynamic shared memory: 228 KB per SM, 1 KB of it reserved per CTA
    const int fixed = (int)sizeof(Stage) * D + 256;
    const int dyn = std::max(0, (228 * 1024) / ctas - 1024 - fixed);
    CHECK(cudaFuncSetAttribute(traffic_bulk<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn));
    int resident = 0;
    CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, traffic_bulk<D>, kBlock, dyn));
    const float ms = time_ms([&] { traffic_bulk<D><<<grid, kBlock, dyn>>>(b); });
    CHECK(cudaGetLastError());
    printf("(b) bulk-copy ring   D=%d  %d CTAs/SM (resident %d)  %.4f ms  %.2f TB/s (125 B/env)\n", D, ctas, resident, ms, 125.0 * kEnvs / (ms * 1e-3) / 1e12);
    return 0;
}

int main() {
    Bufs b;
    b.n = kEnvs;
    void *state, *meta, *action, *reward, *done;
    CHECK(cudaMalloc(&state, kEnvs * 48)); CHECK(cudaMalloc(&meta, kEnvs * 4)); CHECK(cudaMalloc(&action, kEnvs * 16));
    CHECK(cudaMalloc(&reward, kEnvs * 4)); CHECK(cudaMalloc(&done, kEnvs));
    CHECK(cudaMemset(state, 0, kEnvs * 48)); CHECK(cudaMemset(meta, 0, kEnvs * 4)); CHECK(cudaMemset(action, 0, kEnvs * 16));
    b.state = (float4*)state; b.meta = (uint32_t*)meta; b.action = (const float4*)action; b.reward = (float*)reward; b.done = (uint8_t*)done;
    const int grid = (int)(kEnvs / kBlock);
    cudaDeviceProp prop;
    CHECK(cudaGetDeviceProperties(&prop, 0));
    printf("%s, %d SMs, %d envs, 125 B per env\n", prop.name, prop.multiProcessorCount, (int)kEnvs);
    {   // a device-to-device copy of the same byte count, for scale
        void* big;
        const size_t half = (size_t)125 * kEnvs / 2;
        CHECK(cudaMalloc(&big, 2 * half));
        const float ms = time_ms([&] { cudaMemcpyAsync((char*)big + half, big, half, cudaMemcpyDeviceToDevice); });
        printf("cudaMemcpyAsync D2D  %.1f MB read + written  %.4f ms  %.2f TB/s\n", 2 * half / 1e6, ms, 2 * half / (ms * 1e-3) / 1e12);
        CHECK(cudaFree(big));
    }
    const float ms = time_ms([&] { traffic_direct<<<grid, kBlock>>>(b); });
    CHECK(cudaGetLastError());
    printf("(a) one thread / env  %.4f ms  %.2f TB/s (125 B/env)\n", ms, 125.0 * kEnvs / (ms * 1e-3) / 1e12);
    for (int ctas : {4, 6, 8}) {
        if (run_bulk<2>(b, grid, ctas) || run_bulk<3>(b, grid, ctas)) return 1;
        if (ctas < 8 && run_bulk<4>(b, grid, ctas)) return 1;
    }
    CHECK(cudaDeviceSynchronize());
    return 0;
}
