// tools/fft_lat.cu — development microbenchmark: LATENCY of the FFT passes for a lone warp (2 groups) per SM, per pass.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "ep_step.cuh"
using namespace tac;
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

template <int NT>
__global__ void __launch_bounds__(NT) lat_kernel(const cplx* g_wT, int reps, long long* times, uint64_t* sink) {
    constexpr int N = 512, M = 256, NG = NT / 16;
    extern __shared__ __align__(16) unsigned char raw[];
    cplx* wT = reinterpret_cast<cplx*>(raw);
    cplx* S = wT + tab_len(N);
    uint32_t* dig = reinterpret_cast<uint32_t*>(S + NG * M);                     // [NG][2][M]: 2 cached digit levels per group
    uint64_t* acc = reinterpret_cast<uint64_t*>(dig + NG * 2 * M);
    const int tid = threadIdx.x, grp = tid >> 4, t = tid & 15;
    for (int i = tid; i < tab_len(N); i += NT) wT[i] = g_wT[i];
    for (int i = tid; i < NG * 2 * M; i += NT) dig[i] = (i * 2654435761u) & 0x0FFF0FFFu;
    for (int i = tid; i < NG * N; i += NT) acc[i] = i * 0x9E3779B97F4A7C15ull;
    __syncthreads();
    const DecompFast dc = make_decomp_fast(12, 3);
    cplx* Sg = S + grp * M; uint32_t* dg = dig + grp * 2 * M; uint64_t* ag = acc + grp * N;
    long long tsum[6] = {0, 0, 0, 0, 0, 0};
    for (int r = 0; r < reps; r++) {
        long long t0 = clock64();
        grp_decomp_fwd1<EpCfg<512, 4, 3, 1>>(t, 0, [&](int jj, uint64_t& x0, uint64_t& x1) { rot_diff_pair<N>(ag, jj, (r * 37 + 5) & 1023, x0, x1); }, dc, dg, Sg);
        __syncwarp();
        long long t1 = clock64();
        fft_fwd_pass2<N>(t, wT, Sg);
        __syncwarp();
        long long t2 = clock64();
        fft_fwd_pass1<N>(t, [&](int jj, double& a, double& b) { unpack_digits(dg[jj], dc, a, b); }, Sg);
        __syncwarp();
        long long t3 = clock64();
        fft_inv_passA<N>(t, wT, Sg);
        __syncwarp();
        long long t4 = clock64();
        fft_inv_passB<N>(t, Sg, [&](int jj, double re, double im) { ag[jj] += f64_to_torus(re * 1e-3); ag[jj + M] += f64_to_torus(im * 1e-3); });
        __syncwarp();
        long long t5 = clock64();
        tsum[0] += t1 - t0; tsum[1] += t2 - t1; tsum[2] += t3 - t2; tsum[3] += t4 - t3; tsum[4] += t5 - t4;
    }
    if (tid == 0 && blockIdx.x == 0) for (int i = 0; i < 5; i++) times[i] = tsum[i];
    if (tid == 0) sink[blockIdx.x] = acc[5] + (uint64_t)(int64_t)S[3].x + dig[7];
}
template <int NT> void run(const cplx* wT, int reps) {
    long long* times; uint64_t* sink; CK(cudaMalloc(&times, 64)); CK(cudaMalloc(&sink, 148 * 8));
    const size_t smem = (size_t)tab_len(512) * 16 + (NT / 16) * (4096 + 2048 + 4096);     // wT, then per group S, 2 digit levels, acc
    CK(cudaFuncSetAttribute(lat_kernel<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    lat_kernel<NT><<<148, NT, smem>>>(wT, reps, times, sink); CK(cudaDeviceSynchronize());
    long long h[5]; CK(cudaMemcpy(h, times, sizeof(h), cudaMemcpyDeviceToHost));
    cudaFuncAttributes fa; CK(cudaFuncGetAttributes(&fa, lat_kernel<NT>));
    printf("warps/SM=%2d regs=%3d  cycles per call:  decomp+fwd1 %6.0f   fwd2 %6.0f   fwd1(cached digits) %6.0f   invA %6.0f   invB+acc %6.0f\n", NT / 32, fa.numRegs,
           (double)h[0] / reps, (double)h[1] / reps, (double)h[2] / reps, (double)h[3] / reps, (double)h[4] / reps);
}
int main(int argc, char** argv) {
    const int reps = argc > 1 ? atoi(argv[1]) : 2000;
    std::vector<cplx> wT(tab_len(512)); build_wT(512, wT.data());
    cplx* d_wT; CK(cudaMalloc(&d_wT, wT.size() * 16)); CK(cudaMemcpy(d_wT, wT.data(), wT.size() * 16, cudaMemcpyHostToDevice));
    run<32>(d_wT, reps); run<64>(d_wT, reps); run<128>(d_wT, reps); run<256>(d_wT, reps);
    return 0;
}
