// Knock-out timing of the SHIPPED cluster kernel (results are wrong with any knock-out; timing only): -DWLM_KO=<bits>
//   1 no raw wait / TMA re-arm   2 no wait for "P full"   4 no wait for "P free"   8 no mel arithmetic   16 no output pass
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -DWLM_KO=.. -I whisper_context_biasing_b200/csrc -I include -o tools/fused_ko_N tools/fused_ko.cu
#include <cuda_runtime.h>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include "logmel_fused.cuh"
using namespace wlm;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e), __FILE__, __LINE__); exit(1);} } while (0)

int main(int argc, char** argv) {
#ifndef KO_MELS
#define KO_MELS 80
#endif
    const int B = argc > 1 ? atoi(argv[1]) : 242, M = KO_MELS;
    // a triangular bank with the structure of the 80-mel Whisper bank is not needed for timing: build the real one
    std::vector<float> dense(201 * M, 0.f);
    {   // Slaney bank (same formulas as feature_extraction.py), float32
        auto hz2mel = [](double f) { return f >= 1000.0 ? 15.0 + log(f / 1000.0) * (27.0 / log(6.4)) : 3.0 * f / 200.0; };
        auto mel2hz = [](double m) { return m >= 15.0 ? 1000.0 * exp((log(6.4) / 27.0) * (m - 15.0)) : 200.0 * m / 3.0; };
        std::vector<double> edges(M + 2);
        for (int i = 0; i < M + 2; ++i) edges[i] = mel2hz(hz2mel(0.0) + (hz2mel(8000.0) - hz2mel(0.0)) * i / (M + 1));
        for (int k = 0; k < 201; ++k)
            for (int m = 0; m < M; ++m) {
                const double f = 8000.0 * k / 200.0;
                const double dn = (f - edges[m]) / (edges[m + 1] - edges[m]), up = (edges[m + 2] - f) / (edges[m + 2] - edges[m + 1]);
                const double t = fmax(0.0, fmin(dn, up));
                dense[k * M + m] = (float)(t * 2.0 / (edges[m + 2] - edges[m]));
            }
    }
    MelSparse sp;
    memset(&sp, 0, sizeof(sp));
    for (int k = 0; k < kNFreq + 3; ++k) sp.lo[k] = -1;
    int prev = -1;
    for (int k = 0; k < kNFreq; ++k) {
        int idx[2], n = 0;
        for (int m = 0; m < M && n < 2; ++m) if (dense[k * M + m] != 0.f) idx[n++] = m;
        if (n == 0) sp.lo[k] = prev;
        else if (n == 2) { sp.lo[k] = idx[0]; sp.w_lo[k] = dense[k * M + idx[0]]; sp.w_hi[k] = dense[k * M + idx[1]]; }
        else if (idx[0] == 0 && prev == -1) { sp.lo[k] = -1; sp.w_hi[k] = dense[k * M]; }
        else { sp.lo[k] = idx[0]; sp.w_lo[k] = dense[k * M + idx[0]]; }
        prev = sp.lo[k];
    }
    static fused::Tables h;
    int variant = 0;
    if (fused::build_tables(sp, M, &h, &variant) != 0 || variant != KO_MELS) { printf("table build failed (variant %d)\n", variant); return 1; }
    fused::Tables* d;
    CK(cudaMalloc(&d, sizeof(h))); CK(cudaMemcpy(d, &h, sizeof(h), cudaMemcpyHostToDevice));
    float *pcm, *out, *gmax;
    CK(cudaMalloc(&pcm, (size_t)B * 480000 * 4)); CK(cudaMalloc(&out, (size_t)B * M * 3000 * 4)); CK(cudaMalloc(&gmax, (size_t)(B + 148 * 16 * 8) * 4));
    std::vector<float> hp(480000);
    for (int i = 0; i < 480000; ++i) hp[i] = 0.1f * sinf(0.37f * i) + 0.05f * sinf(0.011f * i * i * 1e-3f);
    for (int b = 0; b < B; ++b) CK(cudaMemcpy(pcm + (size_t)b * 480000, hp.data(), 480000 * 4, cudaMemcpyHostToDevice));
    #ifndef KO_KERNEL_MELS
#define KO_KERNEL_MELS KO_MELS
#endif
    auto fn = fused::logmel_cluster_kernel<KO_KERNEL_MELS, false, float, false>;   // 0 = the table-driven mel stage
    CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, fused::kSmemBytes));
    cudaLaunchConfig_t cfg; cudaLaunchAttribute at[2];
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(fused::kCluster * 148); cfg.blockDim = dim3(fused::kThreads); cfg.dynamicSmemBytes = fused::kSmemBytes;
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = fused::kCluster; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization; at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 2;
    int maxc = 0;
    CK(cudaOccupancyMaxActiveClusters(&maxc, fn, &cfg));
    ClipArgs a;
    memset(&a, 0, sizeof(a));
    a.pcm = pcm; a.row_stride = 480000; a.dense_len = 480000; a.pcm_format = WLM_PCM_F32; a.n_mels = M; a.B = B;
    a.out = out; a.gmax = gmax; a.out_format = WLM_OUT_F32;
    cfg.gridDim = dim3(fused::kCluster * (B < maxc ? B : maxc));
    a.n_workers = B < maxc ? B : maxc;
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) CK(cudaLaunchKernelEx(&cfg, fn, a, h.mel, (const float*)d->win_lane));
    CK(cudaDeviceSynchronize());
    CK(cudaEventRecord(e0));
    for (int i = 0; i < 10; ++i) CK(cudaLaunchKernelEx(&cfg, fn, a, h.mel, (const float*)d->win_lane));
    CK(cudaEventRecord(e1));
    CK(cudaDeviceSynchronize());
    float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
    const double us = ms * 100.0, rounds = (double)B / maxc;
    printf("%s: B=%d clusters=%d: %.1f us per launch, %.2f us per round, %.0f cycles per 64 frames per SM (at 1.965 GHz)\n",
           argv[0], B, maxc, us, us / rounds, us / rounds / 8.0 * 1965.0);
    {   // FNV-1a over the features of the last launch: builds that must agree bit for bit print the same value
        std::vector<unsigned int> ho((size_t)B * M * 3000);
        CK(cudaMemcpy(ho.data(), out, ho.size() * 4, cudaMemcpyDeviceToHost));
        unsigned long long h64 = 1469598103934665603ull;
        for (size_t i = 0; i < ho.size(); ++i) { h64 ^= ho[i]; h64 *= 1099511628211ull; }
        printf("  features fnv64 %016llx\n", h64);
    }
#ifdef WLM_WAITSTAT
    {   // cycles per warp in each kind of wait, averaged over the warps of the launch (last launch)
        const int nw = (int)cfg.gridDim.x * 16;
        std::vector<float> ws((size_t)nw * 8);
        CK(cudaMemcpy(ws.data(), gmax, ws.size() * 4, cudaMemcpyDeviceToHost));
        double acc[5] = {0, 0, 0, 0, 0};
        for (int w = 0; w < nw; ++w) for (int k = 0; k < 5; ++k) acc[k] += ws[(size_t)w * 8 + k];
        printf("  mean cycles per warp: loop %.0f | wait raw %.0f (%.1f%%) P full %.0f (%.1f%%) P free %.0f (%.1f%%) clip maxima %.0f (%.1f%%)\n",
               acc[4] / nw, acc[0] / nw, 100 * acc[0] / acc[4], acc[1] / nw, 100 * acc[1] / acc[4], acc[2] / nw, 100 * acc[2] / acc[4],
               acc[3] / nw, 100 * acc[3] / acc[4]);
        for (int g = 0; g < 16; ++g) {      // by warp index inside the CTA (8 warps per group)
            double a5[5] = {0, 0, 0, 0, 0};
            for (int c = 0; c < (int)cfg.gridDim.x; ++c) for (int k = 0; k < 5; ++k) a5[k] += ws[((size_t)c * 16 + g) * 8 + k];
            printf("  warp %2d: raw %5.1f%%  P full %5.1f%%  P free %5.1f%%  maxima %5.1f%%\n", g, 100 * a5[0] / a5[4], 100 * a5[1] / a5[4],
                   100 * a5[2] / a5[4], 100 * a5[3] / a5[4]);
        }
    }
#endif
    return 0;
}
