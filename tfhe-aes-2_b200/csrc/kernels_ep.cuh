// kernels_ep.cuh — the FFT / external-product kernels (templated on the polynomial size and GLWE dimension):
// poly_fft_kernel, pbs_kernel, pbs_wide_kernel, pbs_merged_kernel, vp_kernel, vp_gather_kernel, cmux_tree_kernel.  Instantiated per shape in kernels_n512.cu / kernels_n1024.cu.
#pragma once
#include <cuda_runtime.h>
#include "ep_step.cuh"

namespace tac {

template <int N> struct LogN { static constexpr int v = (N == 256) ? 8 : (N == 512) ? 9 : (N == 1024) ? 10 : (N == 2048) ? 11 : -1; };

// ================================================================================================ Fourier transform of torus polynomials
// 16 polynomials per CTA (one per 16-thread group).  out[poly][M] in slot order, scaled by `scale`·2^-64.
template <int N>
__global__ void __launch_bounds__(256)
poly_fft_kernel(const uint64_t* __restrict__ polys, size_t npoly, double scale, const cplx* __restrict__ g_wT, cplx* __restrict__ out) {
    constexpr int M = N / 2;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cplx* S = reinterpret_cast<cplx*>(smem_raw);
    cplx* wT = S + 16 * M;
    for (int i = threadIdx.x; i < tab_len(N); i += 256) wT[i] = g_wT[i];
    __syncthreads();
    const int grp = threadIdx.x >> 4, t = threadIdx.x & 15;
    const size_t poly = (size_t)blockIdx.x * 16 + grp;
    if (poly < npoly) key_fft_pass1<N>(t, polys + poly * N, scale, S + grp * M);
    __syncthreads();
    if (poly < npoly) fft_fwd_pass2<N>(t, wT, S + grp * M);
    __syncthreads();
    const size_t base = (size_t)blockIdx.x * 16 * M;
    const size_t lim = npoly * M;
    for (int i = threadIdx.x; i < 16 * M; i += 256)
        if (base + i < lim) out[base + i] = S[i];
}

// ================================================================================================ CMux chain plumbing
template <class C>
struct EpSmem {
    uint64_t* acc; cplx* S; uint32_t* dig; cplx* wT; unsigned char* extra;
    __device__ explicit EpSmem(unsigned char* raw) {
        acc = reinterpret_cast<uint64_t*>(raw);
        S = reinterpret_cast<cplx*>(acc + C::acc_words);
        dig = reinterpret_cast<uint32_t*>(S + C::s_cplx);
        wT = reinterpret_cast<cplx*>(dig + C::dig_words);
        extra = reinterpret_cast<unsigned char*>(wT + tab_len(C::N));
    }
    static constexpr size_t bytes = C::acc_words * 8 + C::s_cplx * 16 + C::dig_words * 4 + (size_t)tab_len(C::N) * 16;
};

// the Fourier-domain accumulators of ep_step_device start at zero (ph_outw clears them again after each step)
template <int SPT, int B, int G>
__device__ __forceinline__ void zero_fourier_acc(cplx (&out)[SPT][B][G]) {
#pragma unroll
    for (int a = 0; a < SPT; a++)
#pragma unroll
        for (int b = 0; b < B; b++)
#pragma unroll
            for (int c = 0; c < G; c++) out[a][b][c] = mk(0.0, 0.0);
}

// one step on the operand whose coefficients jj and jj + N/2 of polynomial `job` are given by coef(job, jj, x0, x1); the
// accumulators receive  acc += GGSW ⊡ operand.
// Ends with a __syncwarp(): the accumulator rows of a job are only touched by the job's own 16-thread group, so the next
// step's decomposition may follow without a CTA barrier.  (Readers of acc from other groups must __syncthreads() first.)
template <class C, int NT, int MAC_DEPTH = 5, class CoefFn>
__device__ __forceinline__ void ep_step_device(int tid, const EpSmem<C>& sm, const cplx* __restrict__ ggsw, CoefFn coef, int base_log,
                                               cplx (&out)[MacCfg<C, NT>::SPT][C::B][C::G]) {
    typedef MacCfg<C, NT> MC;
    static_assert(NT / 16 >= C::JOBS, "one 16-thread group per operand polynomial");
    const int job = tid >> 4, t = tid & 15;
    const bool active = job < C::JOBS;
    cplx g[MAC_DEPTH][C::G];            // key prefetch ring (ep_step.cuh)
    const DecompFast dc = make_decomp_fast(base_log, C::L);
    // (A variant that ping-pongs between two FFT buffers, so that mac(l) and the transforms of level l-1 share one barrier
    // interval — L+1 barriers instead of 2L — measured 3 % SLOWER on B200 (tools/pbs_bench.cu, 123.2 vs 119.4 ms for 6144
    // ciphertexts) and costs 61 KB more shared memory; the single-buffer schedule below is the one that ships.)
    if (active) grp_decomp_fwd1<C>(t, job, [&](int jj, uint64_t& x0, uint64_t& x1) { coef(job, jj, x0, x1); }, dc, sm.dig, sm.S);
    // The first key rows are requested AFTER pass 2 (in flight during the barrier only): pass 2 holds 16 values and 15
    // twiddles, and a ring that is live across it costs registers the FFT needs (measured with the FMA-fused passes:
    // 112.4 ms late vs 121.8 ms early for 6144 ciphertexts).
    __syncwarp();
    if (active) grp_fwd2<C>(t, job, sm.wT, sm.S);
    ph_mac_prefetch<C, MC::NT_MAC, MAC_DEPTH>(tid, C::L, ggsw, g);
    __syncthreads();
    ph_mac<C, MC::NT_MAC, MC::SPT, MAC_DEPTH>(tid, C::L, ggsw, sm.S, out, g);
    if (C::L == 1) ph_outw<C, MC::NT_MAC, MC::SPT>(tid, sm.S, out);         // own slots only: no barrier needed in between
    __syncthreads();
#pragma unroll
    for (int lev = C::L - 1; lev >= 1; lev--) {
        if (active) grp_fwd1<C>(t, job, lev, dc, sm.dig, sm.S);
        __syncwarp();
        if (active) grp_fwd2<C>(t, job, sm.wT, sm.S);
        ph_mac_prefetch<C, MC::NT_MAC, MAC_DEPTH>(tid, lev, ggsw, g);
        __syncthreads();
        ph_mac<C, MC::NT_MAC, MC::SPT, MAC_DEPTH>(tid, lev, ggsw, sm.S, out, g);
        if (lev == 1) ph_outw<C, MC::NT_MAC, MC::SPT>(tid, sm.S, out);
        __syncthreads();
    }
    if (active) grp_inv1<C>(t, job, sm.wT, sm.S);
    __syncwarp();
    if (active) grp_inv2<C>(t, job, sm.S, sm.acc);
    __syncwarp();
}

// [U] glwe_sample_extraction.rs::extract_lwe_sample_from_glwe_ciphertext(.., MonomialDegree(0)); element e of the LWE
template <class C>
__device__ __forceinline__ uint64_t sample_extract_elem(const uint64_t* __restrict__ glwe, int e) {
    if (e == C::K * C::N) return glwe[(size_t)C::K * C::N];
    const int p = e / C::N, j = e - p * C::N;
    const uint64_t* a = glwe + (size_t)p * C::N;
    return (j == 0) ? a[0] : (0ull - a[C::N - j]);
}

// stand-alone form of the sample extraction the PBS / vertical-packing kernels fuse (parity test entry point)
template <int N, int K>
__global__ void sample_extract_kernel(const uint64_t* __restrict__ glwe, size_t n_glwe, uint64_t* __restrict__ out) {
    typedef EpCfg<N, K, 1, 1> C;
    constexpr size_t LW = (size_t)K * N + 1;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n_glwe * LW; idx += (size_t)gridDim.x * blockDim.x) {
        const size_t g = idx / LW;
        out[idx] = sample_extract_elem<C>(glwe + g * C::G * N, (int)(idx - g * LW));
    }
}

// ================================================================================================ PBS (homomorphic_shift_boolean)
// in: small LWE [nct][n+1]; out: big LWE [nct][kN+1] encrypting bit·2·alpha.
// [U] wop_pbs.rs::homomorphic_shift_boolean + bootstrap.rs::{blind_rotate_assign, bootstrap}
// pbs_kernel, pbs_wide_kernel and pbs_merged_kernel differ only in the step.  They share the mod switch, the prologue
// (twiddles, monomial degrees, trivial accumulators), the epilogue (sample extraction) and rot_sm, the monomial degrees of the
// current and the next step, [2][B] ints after the buffers of each shared-memory layout.  Each layout struct places its
// buffers and counts its bytes; the count sets the dynamic shared memory and with it the L1 left for the in-flight key
// loads, which moves the PBS time (DESIGN.md §4).
constexpr size_t kRotSmBytes = 64;          // the rot_sm area of PbsSmem and MergedSmem

// modulus-switched element i of ciphertext ct0 + b (0 for the padding ciphertexts of the last CTA); n1 = n + 1 is the stride
template <int N>
struct PbsModSwitch {
    const uint64_t* lwe_small;
    int nct, n, n1, ct0;
    __device__ __forceinline__ int operator()(int b, int i) const {
        const int ct = ct0 + b;
        if (ct >= nct) return 0;
        uint64_t a = __ldg(lwe_small + (size_t)ct * n1 + i);
        if (i == n) a += (1ull << 62);                             // centre the error for the negacyclic LUT
        return modswitch(a, LogN<N>::v);
    }
};

// twiddle table; rot_sm = (degree of step 0, degree of the body b~); accumulator = trivial GLWE(-alpha in every coefficient) · X^{-b~}
template <class C, int NT, class Smem>
__device__ __forceinline__ void pbs_prologue(int tid, const Smem& sm, const PbsModSwitch<C::N>& switched, uint64_t alpha,
                                             const cplx* __restrict__ g_wT) {
    constexpr int N = C::N, B = C::B;
    for (int i = tid; i < tab_len(N); i += NT) sm.wT[i] = g_wT[i];
    if (tid < B) { sm.rot_sm[tid] = switched(tid, 0); sm.rot_sm[B + tid] = switched(tid, switched.n); }
    __syncthreads();
    for (int idx = tid; idx < (int)C::acc_words; idx += NT) {
        const int b = idx / (C::G * N), rem = idx - b * C::G * N, p = rem / N, j = rem - p * N;
        uint64_t v = 0;
        if (p == C::K) {
            const int s = (j + sm.rot_sm[B + b]) & (2 * N - 1);
            v = (s < N) ? (0ull - alpha) : alpha;
        }
        sm.acc[idx] = v;
    }
    __syncthreads();
}

// sample extraction of the B accumulators into out[set][first + b] (out: [][count][kN+1]) for first + b < count, alpha added to
// the body.  The caller orders the accumulator writes before it.
template <class C, int NT>
__device__ __forceinline__ void pbs_epilogue(int tid, const uint64_t* acc, uint64_t* out, int set, int first, int count, uint64_t alpha) {
    constexpr int LW = C::K * C::N + 1;
    for (int idx = tid; idx < C::B * LW; idx += NT) {
        const int b = idx / LW, e = idx - b * LW, ct = first + b;
        if (ct >= count) continue;
        uint64_t v = sample_extract_elem<C>(acc + (size_t)b * C::G * C::N, e);
        if (e == C::K * C::N) v += alpha;
        out[((size_t)set * count + ct) * LW + e] = v;
    }
}

// The level-by-level schedule: the PBS path for N = 1024, and at N = 512 the bit-identity reference of pbs_merged_kernel and
// pbs_wide_kernel in tools/pbs_bench.cu.  Layout: EpSmem, then rot_sm.
template <class C> struct PbsSmem : EpSmem<C> {
    int* rot_sm;
    __device__ explicit PbsSmem(unsigned char* raw) : EpSmem<C>(raw), rot_sm(reinterpret_cast<int*>(this->extra)) {}
    static constexpr size_t bytes = EpSmem<C>::bytes + kRotSmBytes;
    static_assert(2 * C::B * sizeof(int) <= kRotSmBytes, "rot_sm");
};

template <int N, int K, int L, int B, int NT, int MAC_DEPTH = 5>
__global__ void __launch_bounds__(NT, 1)
pbs_kernel(const uint64_t* __restrict__ lwe_small, int nct, int n, const cplx* __restrict__ bsk, int base_log, uint64_t alpha,
           const cplx* __restrict__ g_wT, uint64_t* __restrict__ out_big) {
    typedef EpCfg<N, K, L, B> C;
    typedef MacCfg<C, NT> MC;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const PbsSmem<C> sm(smem_raw);
    const int tid = threadIdx.x;
    const int ct0 = blockIdx.x * B;
    const PbsModSwitch<N> switched{lwe_small, nct, n, n + 1, ct0};
    pbs_prologue<C, NT>(tid, sm, switched, alpha, g_wT);
    cplx out[MC::SPT][B][C::G];
    zero_fourier_acc(out);
    const size_t ggsw_sz = (size_t)L * C::G * C::G * C::M;
    for (int i = 0; i < n; i++) {
        const int* rot = sm.rot_sm + (i & 1) * B;
        if (tid < B && i + 1 < n) sm.rot_sm[((i + 1) & 1) * B + tid] = switched(tid, i + 1);      // consumed after >= 1 barrier
        ep_step_device<C, NT, MAC_DEPTH>(tid, sm, bsk + ggsw_sz * i,
                              [&](int job, int jj, uint64_t& x0, uint64_t& x1) { rot_diff_pair<N>(sm.acc + (size_t)job * N, jj, rot[job / C::G], x0, x1); },
                              base_log, out);
    }
    __syncthreads();
    pbs_epilogue<C, NT>(tid, sm.acc, out_big, 0, ct0, nct, alpha);
}

// ================================================================================================ PBS, level-parallel variant
// For small batches (per-block latency) the step of pbs_kernel is a chain of dependent phases executed by one 16-thread
// group per polynomial: decompose → L × (forward FFT → MAC) → inverse FFT.  Here the L levels are transformed AT THE SAME
// TIME by L·B·G groups (one FFT buffer per level), the decomposition of a polynomial is split over L groups, and the MAC runs
// once over all L·G key rows with one prefetch ring.  Same arithmetic in the same order as pbs_kernel — bit-identical
// results — but 4 barriers and one FFT latency per step instead of 2L barriers and L FFT latencies.
//   P0  group (part, job): digits of all levels for its share of the coefficient pairs      ── barrier ──
//   P1  group (level, job): forward FFT of that level from the cached digits                 ── barrier ──
//   P2  256 slot threads: out = Σ_{level, p} fft(digits) · BSK row, written to the level-1 buffer   ── barrier ──
//   P3  group (0, job): inverse FFT + torus accumulate                                        ── barrier ──
// Layout: acc [B][G][N], S [L][JOBS][M] (storage index s ↔ level s+1), dig [JOBS][L][M], wT, rot_sm [2][B], then 80 bytes that
// nothing uses: the mbarrier area and alignment pad of the key staging this kernel had before commit 0336db3.  They stay so
// that the kernel keeps the shared-memory size (and so the L1 size) it was measured with.
template <class C> struct WideSmem {
    uint64_t* acc; cplx* S; uint32_t* dig; cplx* wT; int* rot_sm;
    __device__ explicit WideSmem(unsigned char* raw) {
        acc = reinterpret_cast<uint64_t*>(raw);
        S = reinterpret_cast<cplx*>(acc + C::acc_words);
        dig = reinterpret_cast<uint32_t*>(S + (size_t)C::L * C::s_cplx);
        wT = reinterpret_cast<cplx*>(dig + (size_t)C::JOBS * C::L * C::M);
        rot_sm = reinterpret_cast<int*>(wT + tab_len(C::N));
    }
    static constexpr size_t kUnused = 80;
    static constexpr size_t bytes = C::acc_words * 8 + (size_t)C::L * C::s_cplx * 16 + (size_t)C::JOBS * C::L * C::M * 4 +
                                    (size_t)tab_len(C::N) * 16 + 2 * C::B * sizeof(int) + kUnused;
};

template <int N, int K, int L, int B, int NT, int MAC_DEPTH = 5>
__global__ void __launch_bounds__(NT, 1)
pbs_wide_kernel(const uint64_t* __restrict__ lwe_small, int nct, int n, const cplx* __restrict__ bsk, int base_log, uint64_t alpha,
                const cplx* __restrict__ g_wT, uint64_t* __restrict__ out_big) {
    typedef EpCfg<N, K, L, B> C;
    constexpr int JOBS = C::JOBS, NMAC = C::M;
    static_assert(NT / 16 >= L * JOBS, "one 16-thread group per (level, polynomial)");
    static_assert(NT >= NMAC && MAC_DEPTH <= L * C::G, "one MAC thread per frequency slot");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const WideSmem<C> sm(smem_raw);
    const int tid = threadIdx.x;
    const int grp = tid >> 4, t = tid & 15;
    const int part = grp / JOBS, job = grp - part * JOBS;                      // part: share of the pairs in P0, level index in P1
    const bool active = grp < L * JOBS;
    const int ct0 = blockIdx.x * B;
    const PbsModSwitch<N> switched{lwe_small, nct, n, n + 1, ct0};
    pbs_prologue<C, NT>(tid, sm, switched, alpha, g_wT);
    const DecompFast dc = make_decomp_fast(base_log, L);
    const size_t ggsw_sz = (size_t)L * C::G * C::G * C::M;
    constexpr int P = C::M / 16;
    const int m0 = part * P / L, m1 = (part + 1) * P / L;                     // this group's share of the P register rows
    for (int i = 0; i < n; i++) {
        const int* rot = sm.rot_sm + (i & 1) * B;
        const cplx* ggsw = bsk + ggsw_sz * i;
        if (tid < B && i + 1 < n) sm.rot_sm[((i + 1) & 1) * B + tid] = switched(tid, i + 1);      // consumed after >= 1 barrier
        if (i + kL2PrefetchSteps < n) ggsw_l2_prefetch<C>(ggsw + ggsw_sz * kL2PrefetchSteps, tid, NT);
        // ---- P0: digits
        if (active) {
            const uint64_t* poly = sm.acc + (size_t)job * N;
            const int r = rot[job / C::G];
            uint32_t* dj = sm.dig + (size_t)job * L * C::M;
#pragma unroll 2
            for (int m = m0; m < m1; m++) {
                const int jj = t + 16 * m;
                uint32_t w[L];
                uint64_t x0, x1;
                rot_diff_pair<N>(poly, jj, r, x0, x1);
                decompose_pair<L>(x0, x1, dc, w);
#pragma unroll
                for (int s = 0; s < L; s++) dj[(size_t)s * C::M + jj] = w[s];
            }
        }
        __syncthreads();
        // ---- P1: forward FFT of level part+1 of polynomial job; the MAC threads request their first key rows
        cplx g[MAC_DEPTH][C::G];
        if (tid < NMAC) mg_mac_prefetch<C, MAC_DEPTH>(tid, ggsw, g);
        {
            const uint32_t* d = sm.dig + ((size_t)job * L + part) * C::M;
            cplx* Sj = sm.S + ((size_t)part * JOBS + job) * C::M;
            if (active) fft_fwd_pass1<N>(t, [&](int jj, double& a, double& b) { unpack_digits(d[jj], dc, a, b); }, Sj);
            __syncwarp();                          // outside the predicate: a warp may hold one active and one idle group
            if (active) fft_fwd_pass2<N>(t, sm.wT, Sj);
        }
        __syncthreads();
        // ---- P2: Fourier MAC over all L·G key rows; the sums go to the thread's own slot of buffer 0
        if (tid < NMAC) mg_mac<C, MAC_DEPTH, 0>(tid, ggsw, sm.S, g);
        __syncthreads();
        // ---- P3: inverse FFT and accumulate (the groups of part 0)
        if (active && part == 0) grp_inv1<C>(t, job, sm.wT, sm.S);
        __syncwarp();
        if (active && part == 0) grp_inv2<C>(t, job, sm.S, sm.acc);
        __syncthreads();
    }
    pbs_epilogue<C, NT>(tid, sm.acc, out_big, 0, ct0, nct, alpha);
}

// ================================================================================================ PBS, levels merged (throughput path)
// pbs_kernel runs a step as L × (forward FFT → barrier → MAC → barrier) because one FFT buffer per (ciphertext, polynomial)
// is all that fits next to the accumulators.  Here the accumulators LEAVE shared memory.  The 16-thread group of job (b, p)
// is the only writer of accumulator polynomial (b, p) and, apart from the ROTATED reads of the decomposition, its only
// reader; and each of its threads reads and writes the same 32 coefficients in every step (forward pass 1 consumes samples
// t + 16m and t + 16m + M, inverse pass B produces exactly those).  So every thread keeps its 32 coefficients in registers,
// and the copy the rotated reads need lives in the rows of the level-1 FFT buffer, which are dead between the inverse
// transform of one step and the level-1 forward pass of the next.  Shared memory then holds L buffers per job (184 KB for
// L = 3, B = 3), the digits of all levels stay in registers (no digit cache), and a step needs TWO CTA barriers:
//
//   group (b,p):  rotated reads + digits of all L levels | pass 1 × L | pass 2 × L            ── barrier ──
//   slot thread:  Σ over all L·G key rows, one prefetch ring                → sums in buffer 1   ── barrier ──
//   group (b,c):  inverse pass A | pass B + accumulate (registers) + refresh of the rotation copy
//
// The long barrier-free stretch lets the warps drift apart, so the shared-memory bursts of one warp overlap the FP64 work of
// another; the MAC is one contiguous key stream instead of L ramps.  Same arithmetic in the same order as pbs_kernel —
// bit-identical results (tools/pbs_bench.cu prints the same checksum): 98.3 ms against 111.9 ms for 6144 ciphertexts.
// BLOG > 0: the decomposition base log as a compile-time constant (shifts and masks fold; 0.6 %).
// Layout: S [L][JOBS][M] (buffer s ↔ level s+1) with acc [B][G][N], the rotation copy, on buffer 0; wT, rot_sm.
template <class C> struct MergedSmem {
    cplx* S; uint64_t* acc; cplx* wT; int* rot_sm;
    __device__ explicit MergedSmem(unsigned char* raw) {
        S = reinterpret_cast<cplx*>(raw);
        acc = reinterpret_cast<uint64_t*>(raw);
        wT = S + (size_t)C::L * C::s_cplx;
        rot_sm = reinterpret_cast<int*>(wT + tab_len(C::N));
    }
    static constexpr size_t bytes = (size_t)C::L * C::s_cplx * 16 + (size_t)tab_len(C::N) * 16 + kRotSmBytes;
    static_assert(C::acc_words * 8 == C::s_cplx * 16 && 2 * C::B * sizeof(int) <= kRotSmBytes, "layout");
};

template <int N, int K, int L, int B, int NT, int MAC_DEPTH = 4, int BLOG = 0>
__global__ void __launch_bounds__(NT, 1)
pbs_merged_kernel(const uint64_t* __restrict__ lwe_small, int nct, int n, const cplx* __restrict__ bsk, int base_log, uint64_t alpha,
                  const cplx* __restrict__ g_wT, uint64_t* __restrict__ out_big) {
    typedef EpCfg<N, K, L, B> C;
    constexpr int JOBS = C::JOBS, NMAC = C::M, M = C::M, P = M / 16, SUMS = 1;
    static_assert(N == 512, "one DFT-16 per thread and pass");
    static_assert(L >= 2, "the sums use buffer 1, the rotation copy buffer 0");
    static_assert(NT / 16 >= JOBS && NT >= NMAC && MAC_DEPTH <= L * C::G, "thread layout");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const MergedSmem<C> sm(smem_raw);
    const int tid = threadIdx.x;
    const int job = tid >> 4, t = tid & 15;
    const bool active = job < JOBS;
    const int ct0 = blockIdx.x * B;
    const PbsModSwitch<N> switched{lwe_small, nct, n, n + 1, ct0};
    pbs_prologue<C, NT>(tid, sm, switched, alpha, g_wT);
    uint64_t* Rj = sm.acc + (size_t)(active ? job : 0) * N;                    // this group's polynomial (rotation copy)
    cplx* Sjob = sm.S + (size_t)(active ? job : 0) * M;                        // + s·JOBS·M for buffer s
    uint64_t own0[P], own1[P];                                                 // coefficients t + 16m and t + 16m + M
    static_for<0, P>([&](auto mc) { constexpr int m = decltype(mc)::value; own0[m] = Rj[t + 16 * m]; own1[m] = Rj[t + 16 * m + M]; });
    const DecompFast dc = make_decomp_fast(BLOG ? BLOG : base_log, L);
    const size_t ggsw_sz = (size_t)L * C::G * C::G * C::M;
    for (int i = 0; i < n; i++) {
        const int rot = sm.rot_sm[(i & 1) * B + (active ? job / C::G : 0)];
        const cplx* ggsw = bsk + ggsw_sz * i;
        if (tid < B && i + 1 < n) sm.rot_sm[((i + 1) & 1) * B + tid] = switched(tid, i + 1);      // consumed after >= 1 barrier
        if (i + kL2PrefetchSteps < n) ggsw_l2_prefetch<C>(ggsw + ggsw_sz * kL2PrefetchSteps, tid, NT);
        // ---- digits of all levels, in registers
        uint32_t dg[L][P];
        if (active) mg_digits<C>(t, Rj, rot, own0, own1, dc, dg);
        // ---- forward pass 1 of every level; buffer 0 (the rotation copy) is overwritten last, after the whole group has read it
        static_for<0, L>([&](auto ic) {
            constexpr int s = L - 1 - decltype(ic)::value;
            if (s == 0) __syncwarp();
            if (active)
                fft_fwd_pass1_m<N>(t, [&](auto mc, double& a, double& b) { unpack_digits(dg[s][decltype(mc)::value], dc, a, b); },
                                   Sjob + (size_t)s * JOBS * M);
        });
        __syncwarp();
        // ---- forward pass 2 of every level; then the first key rows are requested (in flight during the barrier)
        static_for<0, L>([&](auto ic) {
            constexpr int s = L - 1 - decltype(ic)::value;
            if (active) fft_fwd_pass2<N>(t, sm.wT, Sjob + (size_t)s * JOBS * M);
        });
        cplx g[MAC_DEPTH][C::G];
        if (tid < NMAC) mg_mac_prefetch<C, MAC_DEPTH>(tid, ggsw, g);
        __syncthreads();
        // ---- Fourier MAC over all L·G key rows; a thread reads and writes only its own slot of every buffer
        if (tid < NMAC) mg_mac<C, MAC_DEPTH, SUMS>(tid, ggsw, sm.S, g);
        __syncthreads();
        // ---- inverse transform of the sums; accumulate in registers; refresh the rotation copy
        if (active) fft_inv_passA<N>(t, sm.wT, Sjob + (size_t)SUMS * JOBS * M);
        __syncwarp();
        if (active) mg_inv2<C>(t, Sjob + (size_t)SUMS * JOBS * M, Rj, own0, own1);
        __syncwarp();
    }
    __syncthreads();
    pbs_epilogue<C, NT>(tid, sm.acc, out_big, 0, ct0, nct, alpha);
}

// ================================================================================================ vertical packing
// One CTA evaluates B outputs of one box (= one circuit_bootstrap call).  ggsw_f: [nbox][n_in][L][G][G][M].
// The accumulator starts from init_glwe (CMux-tree result) when given, else from the trivial GLWE of LUT polynomial o.
// Blind rotation uses GGSWs n_in-1 … first_ggsw with X^{-1}, X^{-2}, X^{-4}, …   ([U] wop_pbs.rs::{vertical_packing, blind_rotate_assign})
template <int N, int K, int L, int B, int NT>
__global__ void __launch_bounds__(NT, 1)
vp_kernel(const cplx* __restrict__ ggsw_f, int n_in, int first_ggsw, const uint64_t* __restrict__ lut, size_t lut_stride,
          const uint64_t* __restrict__ init_glwe, int n_out, int base_log, const cplx* __restrict__ g_wT, uint64_t* __restrict__ out) {
    typedef EpCfg<N, K, L, B> C;
    typedef MacCfg<C, NT> MC;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EpSmem<C> sm(smem_raw);
    const int tid = threadIdx.x;
    const int box = blockIdx.y, o0 = blockIdx.x * B;
    for (int i = tid; i < tab_len(C::N); i += NT) sm.wT[i] = g_wT[i];
    for (int idx = tid; idx < (int)C::acc_words; idx += NT) {
        const int b = idx / (C::G * N), rem = idx - b * C::G * N, p = rem / N, j = rem - p * N;
        const int o = o0 + b;
        uint64_t v = 0;
        if (o < n_out) {
            if (init_glwe) v = init_glwe[((size_t)box * n_out + o) * C::G * N + rem];
            else if (p == K) v = lut[(size_t)o * lut_stride + j];
        }
        sm.acc[idx] = v;
    }
    __syncthreads();
    cplx outr[MC::SPT][B][C::G];
    zero_fourier_acc(outr);
    const size_t ggsw_sz = (size_t)L * C::G * C::G * C::M;
    const cplx* gbox = ggsw_f + (size_t)box * n_in * ggsw_sz;
    int deg = 1;
    for (int g = n_in - 1; g >= first_ggsw; g--) {
        const int rot = 2 * N - deg;            // multiply by X^{-deg}
        ep_step_device<C, NT>(tid, sm, gbox + (size_t)g * ggsw_sz,
                              [&](int job, int jj, uint64_t& x0, uint64_t& x1) { rot_diff_pair<N>(sm.acc + (size_t)job * N, jj, rot, x0, x1); }, base_log, outr);
        deg <<= 1;
    }
    __syncthreads();
    pbs_epilogue<C, NT>(tid, sm.acc, out, box, o0, n_out, 0);
}

// Vertical packing over GGSWs picked by index: box b's input g is GGSW ggsw_idx[b·n_in + g] of ggsw_f ([][L][G][G][M]), so
// boxes may share GGSWs (the 4×4-bit boxes of a GF(2^128) product read each operand bit's GGSW 32 times).  No CMux tree
// (n_in <= log2 N): the accumulator starts from the trivial GLWE of LUT polynomial o, and the steps are vp_kernel's.
template <int N, int K, int L, int B, int NT>
__global__ void __launch_bounds__(NT, 1)
vp_gather_kernel(const cplx* __restrict__ ggsw_f, const int32_t* __restrict__ ggsw_idx, int n_in, const uint64_t* __restrict__ lut,
                 size_t lut_stride, int n_out, int base_log, const cplx* __restrict__ g_wT, uint64_t* __restrict__ out) {
    typedef EpCfg<N, K, L, B> C;
    typedef MacCfg<C, NT> MC;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EpSmem<C> sm(smem_raw);
    const int tid = threadIdx.x;
    const int box = blockIdx.y, o0 = blockIdx.x * B;
    for (int i = tid; i < tab_len(C::N); i += NT) sm.wT[i] = g_wT[i];
    for (int idx = tid; idx < (int)C::acc_words; idx += NT) {
        const int b = idx / (C::G * N), rem = idx - b * C::G * N, p = rem / N, j = rem - p * N;
        const int o = o0 + b;
        sm.acc[idx] = (o < n_out && p == K) ? lut[(size_t)o * lut_stride + j] : 0ull;
    }
    __syncthreads();
    cplx outr[MC::SPT][B][C::G];
    zero_fourier_acc(outr);
    const size_t ggsw_sz = (size_t)L * C::G * C::G * C::M;
    const int32_t* gidx = ggsw_idx + (size_t)box * n_in;
    int deg = 1;
    for (int g = n_in - 1; g >= 0; g--) {
        const int rot = 2 * N - deg;            // multiply by X^{-deg}
        ep_step_device<C, NT>(tid, sm, ggsw_f + (size_t)__ldg(gidx + g) * ggsw_sz,
                              [&](int job, int jj, uint64_t& x0, uint64_t& x1) { rot_diff_pair<N>(sm.acc + (size_t)job * N, jj, rot, x0, x1); }, base_log, outr);
        deg <<= 1;
    }
    __syncthreads();
    pbs_epilogue<C, NT>(tid, sm.acc, out, box, o0, n_out, 0);
}

// One CMux-tree layer ([U] wop_pbs.rs::cmux_tree_memory_optimized, evaluated level by level): for every (box, output,
// pair i): node_out[i] = c0 + G ⊡ (c1 − c0) with c0 = node_in[2i], c1 = node_in[2i+1].  leaf != 0: inputs are LUT
// polynomials (trivial GLWEs).  Implemented with the rotation step on a doubled trick: acc = c0, "rot" disabled — the
// difference c1 − c0 is written to a scratch accumulator instead.  One CTA per node (B = 1).
template <int N, int K, int L, int NT>
__global__ void __launch_bounds__(NT, 1)
cmux_tree_kernel(const cplx* __restrict__ ggsw_f, int n_in, int ggsw_idx, const uint64_t* __restrict__ lut, size_t lut_stride,
                 const uint64_t* __restrict__ node_in, int n_nodes_in, int n_out, int base_log, const cplx* __restrict__ g_wT,
                 uint64_t* __restrict__ node_out) {
    typedef EpCfg<N, K, L, 1> C;
    typedef MacCfg<C, NT> MC;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    EpSmem<C> sm(smem_raw);
    uint64_t* diff = reinterpret_cast<uint64_t*>(sm.extra);       // [G][N]  c1 − c0
    const int tid = threadIdx.x;
    const int pair = blockIdx.x, o = blockIdx.y, box = blockIdx.z;
    const int n_pairs = n_nodes_in / 2;
    for (int i = tid; i < tab_len(C::N); i += NT) sm.wT[i] = g_wT[i];
    for (int idx = tid; idx < C::G * N; idx += NT) {
        uint64_t c0, c1;
        if (node_in) {
            const uint64_t* base = node_in + (((size_t)box * n_out + o) * n_nodes_in + 2 * pair) * C::G * N;
            c0 = base[idx]; c1 = base[(size_t)C::G * N + idx];
        } else {
            const int p = idx / N, j = idx - p * N;
            const uint64_t* lp = lut + (size_t)o * lut_stride + (size_t)(2 * pair) * N;
            c0 = (p == K) ? lp[j] : 0ull; c1 = (p == K) ? lp[N + j] : 0ull;
        }
        sm.acc[idx] = c0; diff[idx] = c1 - c0;
    }
    __syncthreads();
    cplx outr[MC::SPT][1][C::G];
    zero_fourier_acc(outr);
    const size_t ggsw_sz = (size_t)L * C::G * C::G * C::M;
    const cplx* ggsw = ggsw_f + ((size_t)box * n_in + ggsw_idx) * ggsw_sz;
    ep_step_device<C, NT>(tid, sm, ggsw, [&](int job, int jj, uint64_t& x0, uint64_t& x1) { x0 = diff[(size_t)job * N + jj]; x1 = diff[(size_t)job * N + jj + N / 2]; },
                          base_log, outr);
    __syncthreads();
    uint64_t* dst = node_out + (((size_t)box * n_out + o) * n_pairs + pair) * C::G * N;
    for (int idx = tid; idx < C::G * N; idx += NT) dst[idx] = sm.acc[idx];
}

}  // namespace tac
