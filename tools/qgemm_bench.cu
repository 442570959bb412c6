// Stand-alone timing of the quarter GEMM (development aid): build variants with -D switches and
// compare them in one gpurun call.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 [-DQS_DBG_NOSTORE ...] -o qgemm_bench \
//        tools/qgemm_bench.cu quantum_systems_b200/csrc/quarter_gemm.cu quantum_systems_b200/csrc/core.cu
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "../include/qsb200.h"

#ifdef QS_DBG_PHASE_CLOCKS
// exported by quarter_gemm.cu in a -DQS_DBG_PHASE_CLOCKS build only
extern "C" int qs_dbg_phase_clocks(unsigned long long* hist, unsigned long long* sum, unsigned long long* count,
                                   int reset);
constexpr int kPhaseBins = 256, kPhaseBinClk = 256;
#endif

#define CK(x)                                                                        \
    do {                                                                             \
        cudaError_t e = (x);                                                         \
        if (e != cudaSuccess) {                                                      \
            printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__);        \
            return 1;                                                                \
        }                                                                            \
    } while (0)
#define QK(x)                                                                        \
    do {                                                                             \
        if ((x) != 0) {                                                              \
            printf("qs error: %s (line %d)\n", qs_last_error(), __LINE__);           \
            return 1;                                                                \
        }                                                                            \
    } while (0)

int main(int argc, char** argv) {
    const char* tag = argc > 1 ? argv[1] : "variant";
    std::vector<int> sizes;
    for (int i = 2; i < argc; ++i) sizes.push_back(atoi(argv[i]));
    if (sizes.empty()) sizes = {128};
    for (int n : sizes) {
        const int64_t X = (int64_t)n * n * n, K = n, W = n;
        double *A, *M, *out, *image;
        CK(cudaMalloc(&A, X * K * 8));
        CK(cudaMalloc(&out, X * W * 8));
        CK(cudaMalloc(&M, K * W * 8));
        std::vector<double> hm(K * W);
        for (auto& v : hm) v = rand() / (double)RAND_MAX - 0.5;
        CK(cudaMemcpy(M, hm.data(), K * W * 8, cudaMemcpyHostToDevice));
        CK(cudaMemset(A, 0, X * K * 8));
        // a cheap non-trivial fill of A
        std::vector<double> ha(1 << 20);
        for (auto& v : ha) v = rand() / (double)RAND_MAX - 0.5;
        for (int64_t off = 0; off < X * K; off += (1 << 20)) {
            int64_t cnt = X * K - off < (1 << 20) ? X * K - off : (1 << 20);
            CK(cudaMemcpy(A + off, ha.data(), cnt * 8, cudaMemcpyHostToDevice));
        }
        int64_t ib = 0;
        QK(qs_coeff_image_bytes(K, W, QS_F64, QS_F64, &ib));
        CK(cudaMalloc(&image, ib));
        QK(qs_build_coeff_image(M, QS_F64, W, 1, 0, K, W, QS_F64, image, 0));
        cudaEvent_t e0, e1;
        CK(cudaEventCreate(&e0));
        CK(cudaEventCreate(&e1));
        for (int i = 0; i < 3; ++i) QK(qs_quarter_transform(A, QS_F64, X, K, K, image, QS_F64, W, out, X, 1, 0, 1, 0, X, 0));
        CK(cudaDeviceSynchronize());
        const int reps = 10;
#ifdef QS_DBG_PHASE_CLOCKS
        QK(qs_dbg_phase_clocks(nullptr, nullptr, nullptr, 1));
#endif
        CK(cudaEventRecord(e0));
        for (int i = 0; i < reps; ++i) QK(qs_quarter_transform(A, QS_F64, X, K, K, image, QS_F64, W, out, X, 1, 0, 1, 0, X, 0));
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        ms /= reps;
        printf("{\"variant\":\"%s\",\"n\":%d,\"ms\":%.4f,\"tflops\":%.2f}\n", tag, n, ms, 2.0 * X * K * W / ms * 1e-9);
#ifdef QS_DBG_PHASE_CLOCKS
        {   // per warp tile: clocks from tile start to main loop (waits), main loop, epilogue; histogram bins as
            // {"first clock of the bin": warp tiles}
            std::vector<unsigned long long> hist(3 * kPhaseBins);
            unsigned long long sum[3], count = 0;
            QK(qs_dbg_phase_clocks(hist.data(), sum, &count, 0));
            const char* names[3] = {"start_wait", "main_loop", "epilogue"};
            for (int ph = 0; ph < 3; ++ph) {
                printf("{\"variant\":\"%s\",\"n\":%d,\"phase\":\"%s\",\"warp_tiles\":%llu,\"mean_clk\":%.1f,\"hist\":{",
                       tag, n, names[ph], count, count ? (double)sum[ph] / count : 0.0);
                bool first = true;
                for (int b = 0; b < kPhaseBins; ++b)
                    if (hist[ph * kPhaseBins + b]) {
                        printf("%s\"%d\":%llu", first ? "" : ",", b * kPhaseBinClk, hist[ph * kPhaseBins + b]);
                        first = false;
                    }
                printf("}}\n");
            }
        }
#endif
        cudaFree(A); cudaFree(out); cudaFree(M); cudaFree(image);
    }
    return 0;
}
