// ep_step.cuh — one CMux/external-product step for a CTA that owns B GLWE accumulators, as barrier-separated phases.
//
// Shared-memory objects (per CTA):
//   acc   uint64  [B][G][N]       the B accumulators (G = k+1 polynomials each)
//   S     cplx    [B*G][M]        one FFT buffer per (ciphertext, polynomial); reused for the MAC output
//   dig   uint32  [B*G][L-1][M]   decomposition digits of levels 1..L-1 of this step (level L is consumed at once),
//                                 samples (jj, jj+M) packed as 16-bit fields digit + B/2
//   wT    cplx    [N]             twiddle tables of both directions (ep_core.cuh)
// Per-thread registers that live across the phases of one step: out[SPT][B][G] (Fourier-domain accumulators of the
// frequency slots this thread owns).
//
// Work split: one 16-thread group (half a warp) owns one operand polynomial "job" = (ciphertext b, polynomial p): it
// decomposes it, runs its forward FFTs, later its inverse FFT and the accumulator update.  All of that touches only the
// group's own rows of acc / dig / S, so inside a group a __syncwarp() orders the passes.  Only the Fourier-domain
// multiply-accumulate crosses groups (thread τ reads slot τ of every job), so a step needs just two CTA barriers per level:
//
//   group:  decomp + fwd1(L) | fwd2        ── barrier ──  all: mac(L)     ── barrier ──
//   group:  fwd1(l) | fwd2                 ── barrier ──  all: mac(l)     ── barrier ──      l = L-1 … 1   (mac(1) also writes out)
//   group:  inv1 | inv2 |                                                                     ( | = __syncwarp )
// Both the CUDA kernels (kernels_ep.cuh) and the CPU emulation (tests/cpu/ep_emul.cpp) follow this order.
// pbs_merged_kernel runs the L levels of a step in ONE barrier interval (accumulators in registers): see the mg_* functions.
// pbs_wide_kernel shares their one-pass MAC over all L·G key rows (mg_mac_prefetch, mg_mac).
#pragma once
#include "ep_core.cuh"


#include <cmath>

namespace tac {

// Key loads take the read-only path (ld.global.nc); cache hints on top of it measured no different (DESIGN.md §4).
TAC_HD cplx ldg_key(const cplx* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

template <int N_, int K_, int L_, int B_>
struct EpCfg {
    static constexpr int N = N_, K = K_, L = L_, B = B_, G = K_ + 1, M = N_ / 2, JOBS = B_ * (K_ + 1);
    static constexpr size_t acc_words = (size_t)B_ * (K_ + 1) * N_;
    static constexpr size_t s_cplx = (size_t)B_ * (K_ + 1) * (N_ / 2);
    static constexpr size_t dig_words = (size_t)B_ * (K_ + 1) * (L_ > 1 ? L_ - 1 : 0) * (N_ / 2);
};
constexpr int floor_pow2(int x) { int p = 1; while (p * 2 <= x) p *= 2; return p; }
template <class C, int NT>
struct MacCfg {
    static constexpr int NT_MAC = floor_pow2(NT) < C::M ? floor_pow2(NT) : C::M;
    static constexpr int SPT = C::M / NT_MAC;
};

// group phase 1 of a step: decompose the operand polynomial `job` (coef(jj, x0, x1) yields its coefficients jj and jj + M),
// keep the digits of levels 1..L-1 in dig, and run forward-FFT pass 1 on the level-L digits straight from registers.
template <class C, class CoefFn>
TAC_HD void grp_decomp_fwd1(int t, int job, CoefFn coef, const DecompFast& dc, uint32_t* __restrict__ dig, cplx* __restrict__ S) {
    uint32_t* dj = dig + (size_t)job * (C::L - 1) * C::M;
    struct Pair { uint64_t x0, x1; };
    fft_fwd_pass1_2ph<C::N>(t, [&](int jj) { Pair p; coef(jj, p.x0, p.x1); return p; },
        [&](int jj, const Pair& p, double& a, double& b) {
            uint32_t w[C::L];
            decompose_pair<C::L>(p.x0, p.x1, dc, w);
#pragma unroll
            for (int s = 0; s + 1 < C::L; s++) dj[(size_t)s * C::M + jj] = w[s];
            unpack_digits(w[C::L - 1], dc, a, b);
        }, S + (size_t)job * C::M);
}
// forward FFT pass 1 of the cached level-`lev` digits (lev < L)
template <class C>
TAC_HD void grp_fwd1(int t, int job, int lev, const DecompFast& dc, const uint32_t* __restrict__ dig, cplx* __restrict__ S) {
    const uint32_t* d = dig + ((size_t)job * (C::L - 1) + (lev - 1)) * C::M;
    fft_fwd_pass1<C::N>(t, [&](int jj, double& a, double& b) { unpack_digits(d[jj], dc, a, b); }, S + (size_t)job * C::M);
}
template <class C>
TAC_HD void grp_fwd2(int t, int job, const cplx* __restrict__ wT, cplx* __restrict__ S) { fft_fwd_pass2<C::N>(t, wT, S + (size_t)job * C::M); }
// out[b][c] += Σ_p fft(digits_{lev,p} of ct b) · GGSW[lev-1][p][c]   at the slots owned by this thread.
// ggsw: Fourier GGSW of this step, [L][G][G][M] slot-ordered (already scaled by 2^-64 / M).
// Key prefetch ring of the MAC: rows 0..MAC_DEPTH-1 of this thread's first slot are requested BEFORE the barrier that
// precedes the MAC (the L2 latency hides behind the barrier wait), row p+MAC_DEPTH is requested while row p is multiplied.
// MAC_DEPTH is a kernel template parameter (register budget: each ring entry is G complex values).
template <class C, int NT_MAC>
TAC_HD void mac_load_row(const cplx* __restrict__ gl, int p, int tau, cplx (&dst)[C::G]) {
#pragma unroll
    for (int c = 0; c < C::G; c++) dst[c] = ldg_key(gl + (size_t)(p * C::G + c) * C::M + tau);
}
template <class C, int NT_MAC, int MAC_DEPTH>
TAC_HD void ph_mac_prefetch(int tid, int lev, const cplx* __restrict__ ggsw, cplx (&g)[MAC_DEPTH][C::G]) {
    if (tid >= NT_MAC) return;
    const cplx* gl = ggsw + (size_t)(lev - 1) * C::G * C::G * C::M;
#pragma unroll
    for (int p = 0; p < MAC_DEPTH && p < C::G; p++) mac_load_row<C, NT_MAC>(gl, p, tid, g[p]);
}
template <class C, int NT_MAC, int SPT, int MAC_DEPTH>
TAC_HD void ph_mac(int tid, int lev, const cplx* __restrict__ ggsw, const cplx* __restrict__ S, cplx (&out)[SPT][C::B][C::G],
                   cplx (&g)[MAC_DEPTH][C::G]) {
    if (tid >= NT_MAC) return;
    const cplx* gl = ggsw + (size_t)(lev - 1) * C::G * C::G * C::M;
#pragma unroll
    for (int it = 0; it < SPT; it++) {
        const int tau = tid + it * NT_MAC;
        if (it > 0) {
#pragma unroll
            for (int p = 0; p < MAC_DEPTH && p < C::G; p++) mac_load_row<C, NT_MAC>(gl, p, tau, g[p]);
        }
#pragma unroll
        for (int p = 0; p < C::G; p++) {
#pragma unroll
            for (int b = 0; b < C::B; b++) {
                const cplx x = S[(size_t)(b * C::G + p) * C::M + tau];
#pragma unroll
                for (int c = 0; c < C::G; c++) cfma(out[it][b][c], x, g[p % MAC_DEPTH][c]);
            }
            if (p + MAC_DEPTH < C::G) mac_load_row<C, NT_MAC>(gl, p + MAC_DEPTH, tau, g[p % MAC_DEPTH]);
        }
    }
}
// Written right after the last ph_mac without a barrier: a thread only reads and writes its own slots of S.
template <class C, int NT_MAC, int SPT>
TAC_HD void ph_outw(int tid, cplx* __restrict__ S, cplx (&out)[SPT][C::B][C::G]) {
    if (tid >= NT_MAC) return;
#pragma unroll
    for (int it = 0; it < SPT; it++) {
        const int tau = tid + it * NT_MAC;
#pragma unroll
        for (int b = 0; b < C::B; b++)
#pragma unroll
            for (int c = 0; c < C::G; c++) {
                S[(size_t)(b * C::G + c) * C::M + tau] = out[it][b][c];
                out[it][b][c] = mk(0.0, 0.0);
            }
    }
}
template <class C>
TAC_HD void grp_inv1(int t, int job, const cplx* __restrict__ wT, cplx* __restrict__ S) { fft_inv_passA<C::N>(t, wT, S + (size_t)job * C::M); }
template <class C>
TAC_HD void grp_inv2(int t, int job, const cplx* __restrict__ S, uint64_t* __restrict__ acc) {
    uint64_t* poly = acc + (size_t)job * C::N;
    fft_inv_passB<C::N>(t, S + (size_t)job * C::M, [&](int jj, double re, double im) {
        poly[jj] += f64_to_torus(re);
        poly[jj + C::M] += f64_to_torus(im);
    });
}

// ------------------------------------------------------------------------------------------------ L2 prefetch of the key stream
// The CTAs of a launch walk the bootstrapping key in step, and the 208 MB key does not fit L2: it streams from HBM once per
// wave, and whichever CTA reaches GGSW i first waits for HBM inside its MAC (then every CTA of the wave waits with it on the
// same lines).  So every CTA asks L2 for a slice of the GGSW of a LATER step while it works on the current one: `slices` CTAs
// (consecutive block indices are co-resident) cover the GGSW between them, one 128-byte line per thread.  Measured on B200:
// blind rotation of 16384 ciphertexts 260.3 → 253.9 ms, of 6144 98.3 → 95.9 ms (distance 1, 2 and 4 steps alike).
#if defined(__CUDACC__)
template <class C>
__device__ __forceinline__ void ggsw_l2_prefetch(const cplx* __restrict__ ggsw, int tid, int nthreads) {
    constexpr int LINES = (int)((size_t)C::L * C::G * C::G * C::M * sizeof(cplx) / 128);
    const int slices = min((int)gridDim.x, 128);
    const int per = min((LINES + slices - 1) / slices, nthreads);
    const int line = (int)(blockIdx.x % slices) * per + tid;
    if (tid < per && line < LINES) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(ggsw) + (size_t)line * 128));
}
#endif
constexpr int kL2PrefetchSteps = 2;          // how many steps ahead

// ------------------------------------------------------------------------------------------------ levels-merged step (pbs_merged_kernel)
// Phase functions of the schedule that keeps the accumulator coefficients of a thread in registers (own0[m], own1[m]:
// coefficients t + 16m and t + 16m + M of the group's polynomial) and the rotation copy `Rj` in the rows of FFT buffer 0.
//
// digits of all L levels of (Rj · X^rot − own): dg[s][m] packs the level-(s+1) digits of samples t + 16m (low half-word) and
// t + 16m + M (high half-word); the rotated loads of a chunk are issued first (cf. rot_diff_pair).  One tie test per chunk:
// a test per coefficient pair (decompose_pair, the form the other kernels use) measured 1.7 % slower here.
template <class C>
TAC_HD void mg_digits(int t, const uint64_t* __restrict__ Rj, int rot, const uint64_t (&own0)[C::M / 16], const uint64_t (&own1)[C::M / 16],
                      const DecompFast& dc, uint32_t (&dg)[C::L][C::M / 16]) {
    constexpr int N = C::N, P = C::M / 16, CH = kLoadChunk;
    constexpr int LOGN = (N == 256) ? 8 : (N == 512) ? 9 : (N == 1024) ? 10 : 11;
    static_for<0, P, CH>([&](auto cc) {
        constexpr int c0 = decltype(cc)::value;
        uint64_t v0[CH], v1[CH];
        uint32_t g0[CH], g1[CH];
        static_for<0, CH>([&](auto kc) {
            constexpr int k = decltype(kc)::value;
            const int jj = t + 16 * (c0 + k);
            const uint32_t s0 = (uint32_t)(jj - rot) & (uint32_t)(2 * N - 1);
            const uint32_t i0 = s0 & (uint32_t)(N - 1), i1 = i0 ^ (uint32_t)(N / 2);
            g0[k] = s0 >> LOGN; g1[k] = g0[k] ^ (i0 >> (LOGN - 1));
            v0[k] = Rj[i0]; v1[k] = Rj[i1];
        });
        // closed-form digits of the whole chunk, ONE tie test per chunk (a branch per pair exposes the latency of the
        // pair's dependent chain every time: in-order issue waits for the predicate)
        uint64_t x0[CH], x1[CH];
        uint32_t probe = 0;
        static_for<0, CH>([&](auto kc) {
            constexpr int k = decltype(kc)::value, m = c0 + k;
            const uint32_t m0 = 0u - g0[k], m1 = 0u - g1[k];
            const uint64_t w0 = ((uint64_t)((uint32_t)(v0[k] >> 32) ^ m0) << 32) | ((uint32_t)v0[k] ^ m0);
            const uint64_t w1 = ((uint64_t)((uint32_t)(v1[k] >> 32) ^ m1) << 32) | ((uint32_t)v1[k] ^ m1);
            x0[k] = (w0 + g0[k]) - own0[m]; x1[k] = (w1 + g1[k]) - own1[m];
            const uint64_t y0 = x0[k] + dc.add, y1 = x1[k] + dc.add;
            static_for<0, C::L>([&](auto sc) {
                constexpr int s = decltype(sc)::value, l = s + 1;
                const uint32_t f0 = (uint32_t)(y0 >> (64 - dc.b * l)) & dc.mask;
                const uint32_t f1 = (uint32_t)(y1 >> (64 - dc.b * l)) & dc.mask;
                dg[s][m] = f0 | (f1 << 16);
                probe |= dg[s][m] - 0x00010001u;
            });
        });
        if (probe & 0x80008000u) {                       // some pair of the chunk may hold an exact tie: replay those exactly
            static_for<0, CH>([&](auto kc) {
                constexpr int k = decltype(kc)::value, m = c0 + k;
                uint32_t pm = 0;
                static_for<0, C::L>([&](auto sc) { pm |= dg[decltype(sc)::value][m] - 0x00010001u; });
                if (pm & 0x80008000u) {
                    const uint64_t p0 = decompose_digits_slow<C::L>(x0[k], dc.b), p1 = decompose_digits_slow<C::L>(x1[k], dc.b);
                    static_for<0, C::L>([&](auto sc) {
                        constexpr int s = decltype(sc)::value;
                        dg[s][m] = ((uint32_t)(p0 >> (16 * s)) & 0xFFFFu) | (((uint32_t)(p1 >> (16 * s)) & 0xFFFFu) << 16);
                    });
                }
            });
        }
    });
}
// The one-pass MAC over all L·G key rows, used by pbs_merged_kernel and pbs_wide_kernel.
// key row r of a step's Fourier GGSW in MAC order: level L first, polynomial p inside
template <class C>
TAC_HD const cplx* mg_row(const cplx* __restrict__ ggsw, int r) { return ggsw + (size_t)((C::L - 1 - r / C::G) * C::G + (r % C::G)) * C::G * C::M; }
template <class C, int MAC_DEPTH>
TAC_HD void mg_mac_prefetch(int tid, const cplx* __restrict__ ggsw, cplx (&g)[MAC_DEPTH][C::G]) {
#pragma unroll
    for (int r = 0; r < MAC_DEPTH; r++) mac_load_row<C, C::M>(mg_row<C>(ggsw, r), 0, tid, g[r]);
}
// slot thread `tid`: Σ over all L·G key rows of the spectra in S[L][JOBS][M] (buffer s ↔ level s+1); the sums replace the
// thread's own slot of buffer `SUMS` (a thread reads and writes only its own slot of every buffer)
template <class C, int MAC_DEPTH, int SUMS>
TAC_HD void mg_mac(int tid, const cplx* __restrict__ ggsw, cplx* __restrict__ S, cplx (&g)[MAC_DEPTH][C::G]) {
    constexpr int ROWS = C::L * C::G;
    cplx out[C::B][C::G];
#pragma unroll
    for (int b = 0; b < C::B; b++)
#pragma unroll
        for (int c = 0; c < C::G; c++) out[b][c] = mk(0.0, 0.0);
#pragma unroll
    for (int r = 0; r < ROWS; r++) {
        const int s = C::L - 1 - r / C::G, p = r % C::G;
#pragma unroll
        for (int b = 0; b < C::B; b++) {
            const cplx x = S[((size_t)s * C::JOBS + b * C::G + p) * C::M + tid];
#pragma unroll
            for (int c = 0; c < C::G; c++) cfma(out[b][c], x, g[r % MAC_DEPTH][c]);
        }
        if (r + MAC_DEPTH < ROWS) mac_load_row<C, C::M>(mg_row<C>(ggsw, r + MAC_DEPTH), 0, tid, g[r % MAC_DEPTH]);
    }
#pragma unroll
    for (int b = 0; b < C::B; b++)
#pragma unroll
        for (int c = 0; c < C::G; c++) S[((size_t)SUMS * C::JOBS + b * C::G + c) * C::M + tid] = out[b][c];
}
// inverse pass B of the sums + accumulate into the thread's coefficients + refresh of the rotation copy
template <class C>
TAC_HD void mg_inv2(int t, const cplx* __restrict__ Ssum, uint64_t* __restrict__ Rj, uint64_t (&own0)[C::M / 16], uint64_t (&own1)[C::M / 16]) {
    fft_inv_passB_m<C::N>(t, Ssum, [&](auto mc, double re, double im) {
        constexpr int m = decltype(mc)::value;
        own0[m] += f64_to_torus(re);
        own1[m] += f64_to_torus(im);
        Rj[t + 16 * m] = own0[m];
        Rj[t + 16 * m + C::M] = own1[m];
    });
}

// Fourier transform of a torus polynomial (keys): 16 threads, buffer S[M]; result left in S in slot order, scaled by `scale`·2^-64.
template <int N>
TAC_HD void key_fft_pass1(int t, const uint64_t* __restrict__ poly, double scale, cplx* __restrict__ S) {
    fft_fwd_pass1<N>(t, [&](int jj, double& a, double& b) {
        a = torus_to_f64(poly[jj]) * scale;
        b = torus_to_f64(poly[jj + N / 2]) * scale;
    }, S);
}

// host-side construction of the twiddle tables (tab_len(N) entries, layout in ep_core.cuh) in extended precision
inline void build_wT(int N, cplx* wT) {
    const int M = N / 2, P = M / 16;
    const long double pi = 3.141592653589793238462643383279502884L;
    for (int i = 0; i < tab_len(N); i++) wT[i] = mk(0.0, 0.0);
    for (int q = 0; q < P; q++) {
        const long double rho = pi / N - 2.0L * pi * (long double)q / M;           // arg ρ_q
        for (int t = 0; t < 16; t++) wT[slot_of(q, t)] = mk((double)cosl(rho * t), (double)sinl(rho * t));
        for (int len = 2; len <= 16; len *= 2)
            for (int k = 0; k < len / 2; k++) {
                const long double ang = rho * (16 / len) - 2.0L * pi * (long double)k / len;
                wT[M + (len / 2 - 1 + k) * P + q] = mk((double)cosl(ang), (double)sinl(ang));
            }
    }
}

}  // namespace tac
