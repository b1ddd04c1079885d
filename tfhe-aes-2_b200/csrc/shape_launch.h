// shape_launch.h — host entry points of the FFT / external-product kernels, one set per (polynomial size, GLWE dimension).
// Each set lives in its own translation unit (kernels_n512.cu, kernels_n1024.cu) so the shapes compile in parallel.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstddef>

namespace tac {

struct KLaunch {
    cudaStream_t stream;
    const double2* wT;      // combined twist/twiddle table of this polynomial size
    int sm_count;
};

struct ShapeOps {
    int N, K;
    // torus polynomials → Fourier slots, scaled by `scale`·2^-64
    cudaError_t (*poly_fft)(const KLaunch&, const uint64_t* polys, size_t npoly, double scale, double2* out);
    // homomorphic_shift_boolean with `levels` BSK levels; cudaErrorInvalidValue if that level count is not instantiated
    cudaError_t (*pbs)(const KLaunch&, int levels, const uint64_t* small, int nct, int n, const double2* bsk, int base_log, uint64_t alpha,
                       uint64_t* out);
    // blind-rotation part of vertical packing (GGSWs n_in-1 … first) with `levels` circuit-bootstrap levels;
    // cudaErrorInvalidValue if that level count is not instantiated
    cudaError_t (*vp)(const KLaunch&, int levels, const double2* ggsw_f, int nbox, int n_in, int first, const uint64_t* lut, size_t lut_stride,
                      const uint64_t* init_glwe, int n_out, int base_log, uint64_t* out);
    // vertical packing with box b's input g read from GGSW ggsw_idx[b·n_in + g] (device array); n_in <= log2 N, else
    // cudaErrorInvalidValue
    cudaError_t (*vp_gather)(const KLaunch&, int levels, const double2* ggsw_f, const int32_t* ggsw_idx, int nbox, int n_in, const uint64_t* lut,
                             size_t lut_stride, int n_out, int base_log, uint64_t* out);
    // one CMux-tree layer
    cudaError_t (*tree)(const KLaunch&, int levels, const double2* ggsw_f, int nbox, int n_in, int ggsw_idx, const uint64_t* lut, size_t lut_stride,
                        const uint64_t* node_in, int n_nodes_in, int n_out, int base_log, uint64_t* node_out);
    // one CMux-with-rotation step per accumulator (test entry point)
    cudaError_t (*cmux_test)(const KLaunch&, int levels, const double2* ggsw_f, const int* rot, int base_log, int n_acc, uint64_t* acc);
    // GLWE [n][(k+1)N] → LWE [n][kN+1], coefficient 0 (test entry point of the fused sample extraction)
    cudaError_t (*sample_extract)(const KLaunch&, const uint64_t* glwe, size_t n, uint64_t* out);
};

const ShapeOps* shape_ops_n512_k4();
const ShapeOps* shape_ops_n1024_k2();

}  // namespace tac
