// Developer microbenchmark: a clock64 timeline of the tcgen05 policy kernel (csrc/copter_policy_tc.cuh built with
// COPTER_POLICY_TC_TRACE) -- for a few CTAs and a few steady-state tiles, when each epilogue warp woke up on the
// layer's `done` barrier, finished its tanh / pack / store work and arrived on `ready`, and when the MMA thread woke
// up and committed.  Answers: where do the ~6900 cycles a tile spends in a CTA go (5 CTAs per SM, 0.32 ms for 2^23
// envs), given that neither the MUFU pipe (61 %) nor the issue slots (59 %) are saturated?
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -fmad=false -DCOPTER_POLICY_TC_TRACE -Igym_copter_b200/csrc
//        -o tools/microbench/policy_tc_trace tools/microbench/policy_tc_trace.cu
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cmath>
#include <cuda_runtime.h>
#include <stdint.h>
#include "copter_policy.cuh"
#include "copter_policy_tc.cuh"

using namespace copter;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)

int main(int argc, char** argv) {
    const int64_t n = argc > 1 ? atoll(argv[1]) : (1ll << 23);
    std::vector<float> h(3 * n * 4), w(64 * 10 + 64 + 64 * 64 + 64 + 4 * 64 + 4);
    srand(1);
    for (auto& v : h) v = (rand() / (float)RAND_MAX - 0.5f) * 2.0f;
    for (auto& v : w) v = (rand() / (float)RAND_MAX - 0.5f) * 0.6f;
    float *state, *wd, *action;
    CK(cudaMalloc(&state, h.size() * 4)); CK(cudaMalloc(&wd, w.size() * 4)); CK(cudaMalloc(&action, n * 16));
    CK(cudaMemcpy(state, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(wd, w.data(), w.size() * 4, cudaMemcpyHostToDevice));
    tc::Args a;
    a.state = state; a.stride = n; a.env_stride = 1; a.n = n;
    a.w1 = wd; a.b1 = wd + 640; a.w2 = wd + 704; a.b2 = wd + 704 + 4096; a.w3 = wd + 704 + 4160; a.b3 = wd + 704 + 4160 + 256;
    a.out_scale = 1.f; a.out_offset = 0.f; a.action = action;
    constexpr auto kernel = tc::copter_mlp_policy_tc_kernel<0, 10, 4>;
    constexpr int smem = (int)sizeof(tc::Smem) + 128;
    CK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    const int grid = (int)((n + tc::kTile - 1) / tc::kTile);          // one CTA per tile: cluster launch control
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    for (int i = 0; i < 3; ++i) kernel<<<grid, tc::kThreads, smem>>>(a);
    CK(cudaDeviceSynchronize());
    cudaEventRecord(e0);
    for (int i = 0; i < 20; ++i) kernel<<<grid, tc::kThreads, smem>>>(a);
    cudaEventRecord(e1); CK(cudaDeviceSynchronize());
    float ms; cudaEventElapsedTime(&ms, e0, e1);
    {   // correctness: a sample of envs against the fp64 evaluation of the same network
        std::vector<float> act(n * 4);
        CK(cudaMemcpy(act.data(), action, n * 16, cudaMemcpyDeviceToHost));
        const float *W1 = w.data(), *B1 = W1 + 640, *W2 = W1 + 704, *B2 = W2 + 4096, *W3 = B2 + 64, *B3 = W3 + 256;
        double worst = 0, mean = 0; int64_t cnt = 0;
        for (int64_t i = 0; i < n; i += (i < 512 || i >= n - 512) ? 1 : 4099) {
            double x[12], h1[64], h2[64];
            for (int j = 0; j < 12; ++j) x[j] = h[((int64_t)(j / 4) * n + i) * 4 + j % 4];
            for (int o = 0; o < 64; ++o) { double s = B1[o]; for (int k = 0; k < 10; ++k) s += W1[o * 10 + k] * x[k]; h1[o] = tanh(s); }
            for (int o = 0; o < 64; ++o) { double s = B2[o]; for (int k = 0; k < 64; ++k) s += W2[o * 64 + k] * h1[k]; h2[o] = tanh(s); }
            for (int o = 0; o < 4; ++o) { double s = B3[o]; for (int k = 0; k < 64; ++k) s += W3[o * 64 + k] * h2[k]; const double e = fabs(tanh(s) - act[i * 4 + o]); worst = e > worst ? e : worst; mean += e; ++cnt; }
        }
        printf("check: max |action - fp64 network| %.5f, mean %.5f over %lld values (bf16 operands: ~1e-2 / 1e-3 expected)\n", worst, mean / cnt, (long long)cnt);
    }
    printf("policy tc kernel (traced build): %.4f ms per launch, %lld envs, grid %d x %d threads, %d B smem\n", ms / 20, (long long)n, grid, tc::kThreads, smem);
#ifdef COPTER_POLICY_TC_TRACE
    static long long tr[tc::kTraceCtas][tc::kTraceTiles][5][32];
    CK(cudaMemcpyFromSymbol(tr, tc::g_trace, sizeof(tr)));
    // events: layer l in 0..2: 3l = woke up on done / (MMA: woke up on ready), 3l+1 = epilogue work done, 3l+2 = arrived / (MMA: committed)
    static long long tc_cta[tc::kTraceCtas][4];
    CK(cudaMemcpyFromSymbol(tc_cta, tc::g_trace_cta, sizeof(tc_cta)));
    for (int c = 0; c < tc::kTraceCtas; ++c) {
        printf("== CTA %d: set-up %lld cycles, tiles %lld cycles (thread 0 done), exit %lld cycles after entry; tile %d began %lld cycles after set-up\n", c * tc::kTraceCtaStep,
               tc_cta[c][1] - tc_cta[c][0], tc_cta[c][2] - tc_cta[c][1], tc_cta[c][3] - tc_cta[c][0], tc::kTraceFirstTile, tr[c][0][4][0] - tc_cta[c][1]);
        for (int r = 0; r + 1 < tc::kTraceTiles; ++r) {
            const long long t0 = tr[c][r][4][0];          // MMA thread woke up for layer 1 of this tile
            printf(" tile %d (cycles since the MMA thread woke up for its layer 1; tile period %lld)\n", r + tc::kTraceFirstTile, tr[c][r + 1][4][0] - t0);
            for (int l = 0; l < 3; ++l) {
                printf("  L%d  mma: wake %6lld commit %6lld |", l + 1, tr[c][r][4][3 * l] - t0, tr[c][r][4][3 * l + 2] - t0);
                for (int wq = 0; wq < 4; ++wq)
                    printf(" w%d: wake %6lld work %6lld arr %6lld |", wq, tr[c][r][wq][3 * l] - t0, tr[c][r][wq][3 * l + 1] - t0, tr[c][r][wq][3 * l + 2] - t0);
                printf("\n");
            }
            for (int l = 0; l < 2; ++l) {
                printf("  L%d chunks (landed/issued):", l + 1);
                for (int wq = 0; wq < 4; ++wq) {
                    printf(" w%d:", wq);
                    for (int q = 0; q < 4; ++q) printf(" %5lld/%5lld", tr[c][r][wq][12 + 8 * l + 2 * q] - t0, tr[c][r][wq][12 + 8 * l + 2 * q + 1] - t0);
                    printf(" |");
                }
                printf("\n");
            }
        }
    }
#endif
    return 0;
}
