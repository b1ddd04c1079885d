// tools/fft_micro.cu — development microbenchmark: how fast do the FFT phases of the external product run on their own,
// as a function of the number of resident warps?  Each 16-thread group loops over forward (digits → pass 1 → pass 2) and
// inverse (pass A → pass B → torus accumulate) transforms on its own shared-memory buffers; occupancy is varied through
// the dynamic shared-memory size.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "ep_step.cuh"
using namespace tac;
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); exit(1); } } while (0)

template <int MODE, int NT, int SYNC>
__global__ void __launch_bounds__(NT) fft_loop(const cplx* g_wT, int reps, uint64_t* sink) {
    constexpr int N = 512, M = 256, NG = NT / 16;
    constexpr bool HAS_S = MODE <= 2, HAS_DIG = MODE != 1, HAS_ACC = MODE >= 1;
    extern __shared__ __align__(16) unsigned char raw[];
    cplx* wT = reinterpret_cast<cplx*>(raw);
    cplx* S = wT + tab_len(N);                                                   // [NG][M]
    uint32_t* dig = reinterpret_cast<uint32_t*>(S + (HAS_S ? NG * M : 0));       // [NG][M]
    uint64_t* acc = reinterpret_cast<uint64_t*>(dig + (HAS_DIG ? NG * M : 0));   // [NG][N]
    const int tid = threadIdx.x, grp = tid >> 4, t = tid & 15;
    for (int i = tid; i < tab_len(N); i += NT) wT[i] = g_wT[i];
    if (HAS_DIG) for (int i = tid; i < NG * M; i += NT) dig[i] = (i * 2654435761u) & 0x0FFF0FFFu;
    if (HAS_ACC) for (int i = tid; i < NG * N; i += NT) acc[i] = i * 0x9E3779B97F4A7C15ull;
    if (HAS_S) for (int i = tid; i < NG * M; i += NT) S[i] = mk(1e-3 * i, -2e-3 * i);
    __syncthreads();
    const DecompFast dc = make_decomp_fast(12, 3);
    cplx* Sg = S + grp * M; uint32_t* dg = dig + grp * M; uint64_t* ag = acc + grp * N;
    const bool active = (SYNC < 2) || grp < NG - 1;
    for (int r = 0; r < reps; r++) {
        if (SYNC) __syncthreads();
        if (MODE == 0 || MODE == 2) {
            if (active) fft_fwd_pass1<N>(t, [&](int jj, double& a, double& b) { unpack_digits(dg[jj], dc, a, b); }, Sg);
            __syncwarp();
            if (active) fft_fwd_pass2<N>(t, wT, Sg);
            __syncwarp();
        }
        if (MODE == 1 || MODE == 2) {
            if (active) fft_inv_passA<N>(t, wT, Sg);
            __syncwarp();
            if (active) fft_inv_passB<N>(t, Sg, [&](int jj, double re, double im) { ag[jj] += f64_to_torus(re * 1e-3); ag[jj + M] += f64_to_torus(im * 1e-3); });
            __syncwarp();
        }
        if (MODE == 3) {      // decomposition only: rot_diff + digits -> dig
            const int rot = (r * 37 + blockIdx.x) & 1023;
            if (active) {
#pragma unroll
                for (int m = 0; m < 16; m++) {
                    const int jj = t + 16 * m;
                    uint32_t w[3];
                    decompose_pair<3>(rot_diff<N>(ag, jj, rot), rot_diff<N>(ag, jj + M, rot), dc, w);
                    dg[jj] = w[0] ^ w[1] ^ w[2];
                }
            }
            __syncwarp();
        }
    }
    __syncthreads();
    if (tid == 0) sink[blockIdx.x] = (HAS_ACC ? acc[5] : 0) + (HAS_S ? (uint64_t)(int64_t)S[3].x : 0) + (HAS_DIG ? dig[7] : 0);
}

template <int MODE, int NT, int SYNC = 0>
void run(const char* name, const cplx* wT, uint64_t* sink, int reps, double peak) {
    constexpr int NG = NT / 16;
    const size_t need = (size_t)tab_len(512) * 16 + (size_t)NG * ((MODE <= 2 ? 4096 : 0) + (MODE != 1 ? 1024 : 0) + (MODE >= 1 ? 4096 : 0));
    for (int want = 1; want <= 8; want++) {
        size_t smem = (227 * 1024 / want) & ~(size_t)1023;
        if (smem > 1024) smem -= 1024;
        if (smem < need) break;
        auto kern = fft_loop<MODE, NT, SYNC>;
        CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int occ; CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, NT, smem));
        cudaFuncAttributes fa; CK(cudaFuncGetAttributes(&fa, kern));
        const int grid = 148 * occ;
        cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
        kern<<<grid, NT, smem>>>(wT, reps, sink); CK(cudaDeviceSynchronize());
        CK(cudaEventRecord(e0)); kern<<<grid, NT, smem>>>(wT, reps, sink); CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
        float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
        const double units = (double)grid * (SYNC == 2 ? NG - 1 : NG) * reps * (MODE == 2 ? 2 : 1);
        printf("%-8s sync=%d NT=%3d regs=%3d ctas/SM=%d warps/SM=%2d  %8.3f ms  %7.1f SM-cycles per transform  nominal-FFT %.2f TF/s (%.3f of peak)\n", name, SYNC, NT, fa.numRegs, occ, occ * NT / 32, ms,
               ms * 1e-3 * 1.965e9 * 148 / units, units * 11776.0 / (ms * 1e-3) / 1e12, units * 11776.0 / (ms * 1e-3) / 1e12 / peak);
    }
}
int main(int argc, char** argv) {
    const int reps = argc > 1 ? atoi(argv[1]) : 2000;
    std::vector<cplx> wT(tab_len(512)); build_wT(512, wT.data());
    cplx* d_wT; CK(cudaMalloc(&d_wT, wT.size() * 16)); CK(cudaMemcpy(d_wT, wT.data(), wT.size() * 16, cudaMemcpyHostToDevice));
    uint64_t* sink; CK(cudaMalloc(&sink, 148 * 8 * 8));
    run<0, 256, 0>("forward", d_wT, sink, reps, 36.8);
    run<0, 256, 1>("forward", d_wT, sink, reps, 36.8);
    run<0, 256, 2>("forward", d_wT, sink, reps, 36.8);
    run<1, 256, 0>("inverse", d_wT, sink, reps, 36.8);
    run<1, 256, 1>("inverse", d_wT, sink, reps, 36.8);
    run<3, 256, 0>("decomp", d_wT, sink, reps, 36.8);
    run<3, 256, 1>("decomp", d_wT, sink, reps, 36.8);
    return 0;
}
