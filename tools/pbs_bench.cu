// tools/pbs_bench.cu — stand-alone timing of the blind-rotation kernels (development tool, not part of the product path).
//
//   nvcc -O3 -std=c++17 -lineinfo -gencode arch=compute_100a,code=sm_100a -I../tfhe-aes-2_b200/csrc -o pbs_bench pbs_bench.cu
//   ./pbs_bench [n_cts=6144] [reps=3] [mask]
//
// Random Fourier-domain BSK and random small LWEs (timing does not depend on the values).  Three configurations run on the
// same inputs; bit i of the optional mask selects configuration i:
//   0  pbs_merged_kernel, the shipped throughput kernel
//   1  pbs_wide_kernel, the shipped latency kernel for small batches
//   2  pbs_kernel, the level-by-level schedule, kept as the bit-identity reference
// The arithmetic of a ciphertext does not depend on the kernel or on how many ciphertexts share a CTA, so all three must
// print the same output checksum.  Reports ms per launch and the fraction of the measured DFMA peak.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <random>
#include "kernels_ep.cuh"

using namespace tac;

#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

__global__ void dfma_peak(double* out, int iters, double m) {
    double a[16];
#pragma unroll
    for (int i = 0; i < 16; i++) a[i] = threadIdx.x + i;
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++) a[i] = fma(a[i], m, 1e-9);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s += a[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
__global__ void checksum_kernel(const uint64_t* p, size_t n, unsigned long long* out) {
    unsigned long long s = 0;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) s += p[i] * (2 * i + 1);
    atomicAdd(out, s);
}

constexpr int N = 512, K = 4, L = 3, n_lwe = 677, BASE_LOG = 12;

struct Bufs { uint64_t* small; cplx* bsk; cplx* wT; uint64_t* out; unsigned long long* sum; int nct; int reps; double peak; };

// the signature shared by the three PBS kernels
typedef void (*PbsKernel)(const uint64_t*, int, int, const cplx*, int, uint64_t, const cplx*, uint64_t*);

void run(const char* name, PbsKernel kern, unsigned grid, int nt, size_t smem, const Bufs& b) {
    CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaFuncAttributes fa; CK(cudaFuncGetAttributes(&fa, kern));
    int occ = 0; CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, nt, smem));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    CK(cudaMemset(b.out, 0, (size_t)b.nct * (K * N + 1) * 8));
    kern<<<grid, nt, smem>>>(b.small, b.nct, n_lwe, b.bsk, BASE_LOG, 1ull << 50, b.wT, b.out);     // warm-up
    CK(cudaDeviceSynchronize());
    float best = 1e30f, tot = 0;
    for (int r = 0; r < b.reps; r++) {
        CK(cudaEventRecord(e0));
        kern<<<grid, nt, smem>>>(b.small, b.nct, n_lwe, b.bsk, BASE_LOG, 1ull << 50, b.wT, b.out);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
        best = ms < best ? ms : best; tot += ms;
    }
    CK(cudaMemset(b.sum, 0, 8));
    checksum_kernel<<<256, 256>>>(b.out, (size_t)b.nct * (K * N + 1), b.sum);
    unsigned long long h; CK(cudaMemcpy(&h, b.sum, 8, cudaMemcpyDeviceToHost));
    const double flop = (double)b.nct * n_lwe * 389120.0;
    printf("%-28s regs=%3d lmem=%4zu smem=%6zu occ=%d  best %8.3f ms  avg %8.3f ms  %6.2f TF/s  frac %.3f  %7.1f PBS/ms  sum=%016llx\n", name, fa.numRegs,
           (size_t)fa.localSizeBytes, smem, occ, best, tot / b.reps, flop / (best * 1e-3) / 1e12, flop / (best * 1e-3) / 1e12 / b.peak, b.nct / best, h);
    CK(cudaEventDestroy(e0)); CK(cudaEventDestroy(e1));
    fflush(stdout);
}

int main(int argc, char** argv) {
    Bufs b;
    b.nct = argc > 1 ? atoi(argv[1]) : 6144;
    b.reps = argc > 2 ? atoi(argv[2]) : 3;
    const unsigned mask = argc > 3 ? (unsigned)strtoul(argv[3], 0, 0) : 0xffffffffu;
    constexpr int M = N / 2, G = K + 1;
    const size_t bsk_n = (size_t)n_lwe * L * G * G * M;
    std::mt19937_64 rng(7);
    std::vector<uint64_t> small((size_t)b.nct * (n_lwe + 1));
    for (auto& v : small) v = rng();
    std::vector<cplx> bsk(bsk_n);
    std::uniform_real_distribution<double> ud(-0.05, 0.05);
    for (auto& v : bsk) { v.x = ud(rng); v.y = ud(rng); }
    std::vector<cplx> wT(tab_len(N)); build_wT(N, wT.data());
    CK(cudaMalloc(&b.small, small.size() * 8)); CK(cudaMemcpy(b.small, small.data(), small.size() * 8, cudaMemcpyHostToDevice));
    CK(cudaMalloc(&b.bsk, bsk_n * sizeof(cplx))); CK(cudaMemcpy(b.bsk, bsk.data(), bsk_n * sizeof(cplx), cudaMemcpyHostToDevice));
    CK(cudaMalloc(&b.wT, wT.size() * sizeof(cplx))); CK(cudaMemcpy(b.wT, wT.data(), wT.size() * sizeof(cplx), cudaMemcpyHostToDevice));
    CK(cudaMalloc(&b.out, (size_t)b.nct * (K * N + 1) * 8));
    CK(cudaMalloc(&b.sum, 8));
    {   // DFMA peak
        double* d; CK(cudaMalloc(&d, 148 * 8 * 256 * 8));
        cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
        double best = 0;
        for (int r = 0; r < 4; r++) {
            CK(cudaEventRecord(e0)); dfma_peak<<<148 * 8, 256>>>(d, 4096, 1.0000001); CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
            float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
            const double tf = 2.0 * 16 * 4096 * 148 * 8 * 256 / (ms * 1e-3) / 1e12;
            if (r) best = tf > best ? tf : best;
        }
        b.peak = best;
        printf("DFMA peak %.2f TFLOP/s; n_cts %d\n", best, b.nct);
    }
    const unsigned grid3 = (unsigned)((b.nct + 2) / 3), grid1 = (unsigned)b.nct;
    if (mask & 1) run("merged B=3 depth=4 blog=12", pbs_merged_kernel<N, K, L, 3, 256, 4, 12>, grid3, 256, MergedSmem<EpCfg<N, K, L, 3>>::bytes, b);
    if (mask & 2) run("wide B=1 NT=256 depth=3", pbs_wide_kernel<N, K, L, 1, 256, 3>, grid1, 256, WideSmem<EpCfg<N, K, L, 1>>::bytes, b);
    if (mask & 4) run("B=3 NT=256 depth=5", pbs_kernel<N, K, L, 3, 256, 5>, grid3, 256, PbsSmem<EpCfg<N, K, L, 3>>::bytes, b);
    return 0;
}
