// ep_core.cuh — the external-product step (CMux with a monomial rotation) as thread-level phases.
//
//   acc(GLWE) += GGSW ⊡ (acc · X^rot − acc)            reference path: [U] tfhe fft64/crypto/{bootstrap,ggsw,wop_pbs}.rs
//
// Every phase is a __host__ __device__ function of (thread id, shared buffers): the CUDA kernels call them between
// __syncthreads(), and tests/cpu/ep_emul.cpp runs the very same functions thread by thread on the CPU, so the index
// arithmetic (FFT passes, swizzles, slot order, rotation, decomposition) is validated without a GPU.
//
// FFT: a negacyclic size-N real transform is a size-M = N/2 complex FFT of (p[j] + i·p[j+M])·e^{iπj/N}.  M = 16·P and
// one FFT is done by 16 threads in two register passes (DFT-P over the stride-16 samples, transpose through shared
// memory, DFT-16).  Both passes of the forward transform are decimation-in-time with the twiddle applied before the add,
// so the twist and the inter-pass twiddle are folded into the butterflies and every butterfly is 6 FMAs (see bfly_r).
// The Fourier "slot" order produced by the forward transform is arbitrary but fixed; the Fourier-domain keys are
// produced by the same forward routine, all Fourier-domain work is pointwise, and the inverse transform consumes the
// same order.
//
//   slot σ = q·16 + (r ^ (q & 15))  holds frequency  f = q + P·r        (q < P, r < 16)
#pragma once
#include "tac_common.h"
#include <cmath>
#include <cstring>
#include <type_traits>

namespace tac {

#if defined(__CUDACC__)
typedef double2 cplx;
#else
struct alignas(16) cplx { double x, y; };
#endif

TAC_HD cplx mk(double x, double y) { cplx r; r.x = x; r.y = y; return r; }
TAC_HD cplx cmul(cplx a, cplx b) { return mk(fma(-a.y, b.y, a.x * b.x), fma(a.y, b.x, a.x * b.y)); }
TAC_HD cplx cmul_conj(cplx a, cplx b) { return mk(fma(a.y, b.y, a.x * b.x), fma(-a.x, b.y, a.y * b.x)); }   // a * conj(b)
// o += a·b.  The order of the four FMAs is part of the contract: every MAC (ph_mac, and mg_mac, which pbs_merged_kernel and
// pbs_wide_kernel share) accumulates in exactly this order, so all of them produce the same words.
TAC_HD void cfma(cplx& o, cplx a, cplx b) {
    o.x = fma(a.x, b.x, o.x); o.x = fma(-a.y, b.y, o.x);
    o.y = fma(a.y, b.x, o.y); o.y = fma(a.x, b.y, o.y);
}

// 2^52 + f for a small unsigned integer f, without an int→double conversion instruction
TAC_HD double u32_magic(uint32_t f) {
#if defined(__CUDA_ARCH__)
    return __hiloint2double(0x43300000, (int)f);
#else
    const uint64_t bits = 0x4330000000000000ull | (uint64_t)f;
    double d; memcpy(&d, &bits, 8); return d;
#endif
}

// cos(2πk/128), k = 0..32 (first quadrant; the rest by symmetry).  On the device the table sits in constant memory: with
// k a compile-time constant after unrolling, a DFMA/DMUL takes the entry straight from the constant bank (c[bank][imm])
// instead of materialising the 64-bit immediate with two moves per use.
#define TAC_COS128_TABLE \
    1.0, 0.998795456205172392714771604759100694, 0.995184726672196886244836953109479922, 0.989176509964780973451673738016243064, \
    0.980785280403230449126182236134239037, 0.970031253194543992603984207286100251, 0.956940335732208864935797886980269969, 0.941544065183020778412509402599502357, \
    0.923879532511286756128183189396788287, 0.903989293123443331586200297230537049, 0.881921264348355029712756863660388350, 0.857728610000272069902269984284770137, \
    0.831469612302545237078788377617905757, 0.803207531480644909806676512963141924, 0.773010453362736960810906609758469801, 0.740951125354959091175616897495162730, \
    0.707106781186547524400844362104849039, 0.671558954847018400625376850427421803, 0.634393284163645498215171613225493371, 0.595699304492433343467036528829969890, \
    0.555570233019602224742830813948532874, 0.514102744193221726593693838968815773, 0.471396736825997648556387625905254378, 0.427555093430282094320966856888798534, \
    0.382683432365089771728459984030398867, 0.336889853392220050689253212619147570, 0.290284677254462367636192375817395275, 0.242980179903263889948274162077471118, \
    0.195090322016128267848284868477022241, 0.146730474455361751658850129646717820, 0.098017140329560601994195563888641846, 0.049067674327418014254954976942682658, \
    0.0
#if defined(__CUDACC__)
static __constant__ double c_cos128[33] = {TAC_COS128_TABLE};
#endif
// compile-time loop: f(std::integral_constant<int, I>) for I = BEGIN, BEGIN + STEP, … < END.  The DFT code indexes its
// register arrays and the twiddle table only through these constants, so nothing depends on the optimiser's unrolling
// heuristics (a rolled loop would push the data array into local memory).
template <int BEGIN, int END, int STEP = 1, class F>
TAC_HD void static_for(F&& f) {
    if constexpr (BEGIN < END) {
        f(std::integral_constant<int, BEGIN>{});
        static_for<BEGIN + STEP, END, STEP>(f);
    }
}
template <int K>
TAC_HD double cos128() {
    static_assert(K >= 0 && K <= 32, "first quadrant only");
#if defined(__CUDA_ARCH__) && !defined(TAC_TWIDDLE_IMMEDIATES)
    return c_cos128[K];
#else
    constexpr double tab[33] = {TAC_COS128_TABLE};
    return tab[K];
#endif
}
// multiply by exp(-2πi K/128) (INV = false) or exp(+2πi K/128) (INV = true), K in [0, 64)
template <bool INV, int K>
TAC_HD cplx mul_w128(cplx d) {
    static_assert(K >= 0 && K < 64, "twiddle index");
    if constexpr (K == 0) return d;
    else if constexpr (K == 32) return INV ? mk(-d.y, d.x) : mk(d.y, -d.x);
    else if constexpr (K == 16) { const double c = cos128<16>(); return INV ? mk((d.x - d.y) * c, (d.x + d.y) * c) : mk((d.x + d.y) * c, (d.y - d.x) * c); }
    else if constexpr (K == 48) { const double c = cos128<16>(); return INV ? mk(-(d.x + d.y) * c, (d.x - d.y) * c) : mk((d.y - d.x) * c, -(d.x + d.y) * c); }
    else {
        // cos, sin of 2πK/128
        const double wr = (K < 32) ? cos128<(K < 32 ? K : 0)>() : -cos128<(K >= 32 ? 64 - K : 0)>();
        const double ws = (K < 32) ? cos128<(K < 32 ? 32 - K : 0)>() : cos128<(K >= 32 ? K - 32 : 0)>();
        const double wi = INV ? ws : -ws;
        return mk(fma(-d.y, wi, d.x * wr), fma(d.y, wr, d.x * wi));
    }
}
// cos / sin of 2π·A/128 for any integer A, from the first-quadrant table
template <int A>
TAC_HD double cosq() {
    constexpr int a = ((A % 128) + 128) % 128;
    if constexpr (a <= 32) return cos128<(a <= 32 ? a : 0)>();
    else if constexpr (a <= 64) return -cos128<(a > 32 && a <= 64 ? 64 - a : 0)>();
    else if constexpr (a <= 96) return -cos128<(a > 64 && a <= 96 ? a - 64 : 0)>();
    else return cos128<(a > 96 ? 128 - a : 0)>();
}
template <int A> TAC_HD double sinq() { return cosq<A - 32>(); }

// Radix-2 butterfly with the twiddle applied BEFORE the add (decimation in time), fused:
//     (u, w) ← (u + T·w, u − T·w)        a = u + T·w in 4 FMAs, u − T·w = 2u − a in 2 FMAs
// (a separate complex multiply followed by an add and a subtract costs 2 DMUL + 2 DFMA + 4 DADD).  T = exp(2πi·A/128)
// is a compile-time constant taken from the constant bank, or a run-time value (lane-dependent twiddles).
TAC_HD void bfly_r(cplx& u, cplx& w, const cplx T) {
    const double ax = fma(-T.y, w.y, fma(T.x, w.x, u.x));
    const double ay = fma(T.y, w.x, fma(T.x, w.y, u.y));
    w = mk(fma(2.0, u.x, -ax), fma(2.0, u.y, -ay));
    u = mk(ax, ay);
}
template <int A>
TAC_HD void bfly_c(cplx& u, cplx& w) {
    constexpr int a = ((A % 128) + 128) % 128;
    if constexpr (a == 0) { const cplx x = u; u = mk(x.x + w.x, x.y + w.y); w = mk(x.x - w.x, x.y - w.y); }
    else if constexpr (a == 64) { const cplx x = u; u = mk(x.x - w.x, x.y - w.y); w = mk(x.x + w.x, x.y + w.y); }
    else if constexpr (a == 32) { const cplx x = u, y = w; u = mk(x.x - y.y, x.y + y.x); w = mk(x.x + y.y, x.y - y.x); }       // T = +i
    else if constexpr (a == 96) { const cplx x = u, y = w; u = mk(x.x + y.y, x.y - y.x); w = mk(x.x - y.y, x.y + y.x); }       // T = −i
    else bfly_r(u, w, mk(cosq<a>(), sinq<a>()));
}
template <int P> TAC_HD constexpr int bitrev(int i) {
    int r = 0;
    for (int b = 1; b < P; b <<= 1) { r = (r << 1) | (i & 1); i >>= 1; }
    return r;
}
// In-register decimation-in-time DFT over the P values v[bitrev(n)] = x_n, natural order out.  bf(LEN, k, u, w) performs
// the butterfly at position k of a block of size LEN.  Every butterfly multiplies BEFORE it adds, so a geometric scaling
// of the INPUT,  X[k] = Σ_n x_n ρ^n e^{∓2πi nk/P},  costs nothing: the block-LEN twiddle becomes ρ^{P/LEN}·e^{∓2πi k/LEN}.
// That is how the negacyclic twist and the twiddle between the two passes of the forward transform are absorbed.
template <int P, int LEN, class Bf>
TAC_HD void dit_stages(cplx* v, Bf&& bf) {
    constexpr int half = LEN / 2;
    static_for<0, P, LEN>([&](auto sc) {
        static_for<0, half>([&](auto kc) {
            constexpr int s = decltype(sc)::value, k = decltype(kc)::value;
            bf(std::integral_constant<int, LEN>{}, kc, v[s + k], v[s + k + half]);
        });
    });
    if constexpr (LEN < P) dit_stages<P, LEN * 2>(v, bf);
}
// plain inverse DFT (e^{+2πi nk/P}), unnormalised
template <int P> TAC_HD void dft_inv(cplx* v) {
    dit_stages<P, 2>(v, [&](auto lc, auto kc, cplx& u, cplx& w) { bfly_c<128 * decltype(kc)::value / decltype(lc)::value>(u, w); });
}
TAC_HD constexpr int slot_of(int q, int i) { return q * 16 + (i ^ (q & 15)); }

// Transform layout.  Sample j = t + 16m (t < 16 the lane, m < P), frequency f = q + P·r (q < P, r < 16):
//     Z_f = Σ_j z_j e^{iπj/N} e^{-2πi jf/M}
//         = Σ_t e^{-2πi tr/16} · ρ_q^t · A_t(q),      A_t(q) = Σ_m z_{t+16m} · c^m · e^{-2πi mq/P}
//     c = e^{iπ·16/N}  (compile-time),      ρ_q = e^{iπ/N} · e^{-2πi q/M}  (per lane, from a table)
// pass 1 (lane t) computes A_t(·) with the twist folded into its butterflies, pass 2 (lane q) the outer sum with ρ_q folded.
//     slot σ = slot_of(q, r) = q·16 + (r ^ (q & 15))   holds frequency   f = q + P·r
// One table `wT` of N entries serves both directions:
//     wT[slot_of(q, t)]         = ρ_q^t                                    inverse: twiddle between pass A and pass B (conjugated)
//     wT[M + (LEN/2-1+k)·P + q] = ρ_q^{16/LEN} · e^{-2πi k/LEN}            forward pass 2: butterfly twiddles, LEN = 2,4,8,16, k < LEN/2
// Memory-operation order.  All buffers of a CTA are carved from one dynamic shared-memory array, so the compiler must
// assume that a store to one of them may alias a later load from another and keeps them in program order: a loop of the
// form "load – compute – store" is executed strictly one element at a time and exposes the shared-memory latency every
// time (measured: 16 serialised twiddle loads ≈ 400 cycles of a 1550-cycle pass, tools/fft_lat.cu; PBS kernel 119.4 → 113.4 ms).  The passes below are
// therefore written in CHUNKS: all loads of a chunk first, then the arithmetic and the stores of the chunk.
constexpr int kLoadChunk = 4;                 // operand pairs per chunk of the decomposing pass (2, 4, 8, 16 measure the same)
TAC_HD constexpr int tab_len(int N) { return N; }    // entries of wT

// the pass-1 DFT of the forward transform on v[bitrev(m)] = z_{t+16m}: twist c^m folded (see above)
template <int N>
TAC_HD void dft_fwd_twisted(cplx* v) {
    constexpr int P = N / 32, CP = (1024 / N) * P;             // c^P = exp(2πi·CP/128)
    dit_stages<P, 2>(v, [&](auto lc, auto kc, cplx& u, cplx& w) {
        constexpr int LEN = decltype(lc)::value, k = decltype(kc)::value;
        static_assert((CP - 128 * k) % LEN == 0, "twiddle not on the 128-point grid");
        bfly_c<(CP - 128 * k) / LEN>(u, w);
    });
}
// ------------------------------------------------------------------------------------------------ forward, pass 1
// Two-phase source: `load(jj)` fetches whatever the samples jj and jj + M (0 <= jj < M) are made from (its loads are
// batched per chunk), `finish(jj, raw, a, b)` turns it into the two real samples (and may store by-products).
// Thread t (0..15) of the FFT group.
template <int N, class Load, class Finish>
TAC_HD void fft_fwd_pass1_2ph(int t, Load load, Finish finish, cplx* __restrict__ S) {
    constexpr int M = N / 2, P = M / 16;
    constexpr int CH = kLoadChunk;
    cplx v[P];
    static_for<0, P, CH>([&](auto cc) {
        constexpr int c0 = decltype(cc)::value;
        decltype(load(0)) raw[CH];
        static_for<0, CH>([&](auto kc) { constexpr int k = decltype(kc)::value; raw[k] = load(t + 16 * (c0 + k)); });
        static_for<0, CH>([&](auto kc) {
            constexpr int k = decltype(kc)::value, m = c0 + k;
            double a, b;
            finish(t + 16 * m, raw[k], a, b);
            v[bitrev<P>(m)] = mk(a, b);
        });
    });
    dft_fwd_twisted<N>(v);
    static_for<0, P>([&](auto qc) { constexpr int q = decltype(qc)::value; S[slot_of(q, t)] = v[q]; });
}
// `src(jj, a, b)` yields the real samples jj and jj + M directly (sources without by-product stores)
template <int N, class Src>
TAC_HD void fft_fwd_pass1(int t, Src src, cplx* __restrict__ S) {
    constexpr int M = N / 2, P = M / 16;
    cplx v[P];
    static_for<0, P>([&](auto mc) {
        constexpr int m = decltype(mc)::value;
        double a, b;
        src(t + 16 * m, a, b);
        v[bitrev<P>(m)] = mk(a, b);
    });
    dft_fwd_twisted<N>(v);
    static_for<0, P>([&](auto qc) { constexpr int q = decltype(qc)::value; S[slot_of(q, t)] = v[q]; });
}
// `src(mc, a, b)` receives the register row m as a compile-time constant (std::integral_constant), sample jj = t + 16m:
// for sources that live in per-thread register arrays (pbs_merged_kernel keeps the digits of all levels in registers)
template <int N, class Src>
TAC_HD void fft_fwd_pass1_m(int t, Src src, cplx* __restrict__ S) {
    constexpr int M = N / 2, P = M / 16;
    cplx v[P];
    static_for<0, P>([&](auto mc) {
        constexpr int m = decltype(mc)::value;
        double a, b;
        src(mc, a, b);
        v[bitrev<P>(m)] = mk(a, b);
    });
    dft_fwd_twisted<N>(v);
    static_for<0, P>([&](auto qc) { constexpr int q = decltype(qc)::value; S[slot_of(q, t)] = v[q]; });
}
// ------------------------------------------------------------------------------------------------ forward, pass 2 (in place)
// multiply by exp(2πi·A/128), A a compile-time angle (free for multiples of a quarter turn)
template <int A>
TAC_HD cplx rot128(cplx d) {
    constexpr int a = ((A % 128) + 128) % 128;
    if constexpr (a == 0) return d;
    else if constexpr (a == 32) return mk(-d.y, d.x);
    else if constexpr (a == 64) return mk(-d.x, -d.y);
    else if constexpr (a == 96) return mk(d.y, -d.x);
    else { const double c = cosq<a>(), sn = sinq<a>(); return mk(fma(-d.y, sn, d.x * c), fma(d.y, c, d.x * sn)); }
}
// The 15 twiddles of pass 2 are  ρ_q^{16/LEN} · e^{-2πi k/LEN}.  Only the four powers ρ_q^{8,4,2,1} (the k = 0 entries)
// are read from the table; the others are formed with a compile-time rotation — 8 complex multiplies per pass instead of
// 11 more 16-byte shared-memory loads per thread.  The kernel's load/store unit is its busiest resource (63 % of the
// data-pipe wavefronts) while the FP64 pipe has slack (46 %), so arithmetic is the cheaper currency.
template <int N>
TAC_HD void fft_fwd_pass2(int t, const cplx* __restrict__ wT, cplx* __restrict__ S) {
    constexpr int M = N / 2, P = M / 16;
    const cplx* __restrict__ wF = wT + M;
#pragma unroll
    for (int c2 = 0; c2 < P / 16; c2++) {
        const int q = t + 16 * c2;
        cplx base[4];                      // LEN = 2, 4, 8, 16 at k = 0: table entries 0, 1, 3, 7
        static_for<0, 4>([&](auto ic) { constexpr int i = decltype(ic)::value; base[i] = wF[((1 << i) - 1) * P + q]; });
        cplx v[16];
        static_for<0, 16>([&](auto tc) { constexpr int tt = decltype(tc)::value; v[bitrev<16>(tt)] = S[slot_of(q, tt)]; });
        dit_stages<16, 2>(v, [&](auto lc, auto kc, cplx& u, cplx& w) {
            constexpr int LEN = decltype(lc)::value, k = decltype(kc)::value;
            constexpr int lg = (LEN == 16) ? 3 : (LEN == 8) ? 2 : (LEN == 4) ? 1 : 0;
            bfly_r(u, w, rot128<-128 * k / LEN>(base[lg]));
        });
        static_for<0, 16>([&](auto rc) { constexpr int r = decltype(rc)::value; S[slot_of(q, r)] = v[r]; });
    }
}
// ------------------------------------------------------------------------------------------------ inverse, pass A (in place)
// ρ_q^t for t = 1, 2, 4, 8 are requested together with the data, ahead of the arithmetic (see "Memory-operation order");
// the other powers are formed as products (at most three multiplications deep)
template <int N>
TAC_HD void fft_inv_passA(int t, const cplx* __restrict__ wT, cplx* __restrict__ S) {
    constexpr int M = N / 2, P = M / 16;
#pragma unroll
    for (int c2 = 0; c2 < P / 16; c2++) {
        const int q = t + 16 * c2;
        cplx v[16];
        static_for<0, 16>([&](auto rc) { constexpr int r = decltype(rc)::value; v[bitrev<16>(r)] = S[slot_of(q, r)]; });
        cplx w[16];
        w[1] = wT[slot_of(q, 1)]; w[2] = wT[slot_of(q, 2)]; w[4] = wT[slot_of(q, 4)]; w[8] = wT[slot_of(q, 8)];
        dft_inv<16>(v);
        w[3] = cmul(w[2], w[1]); w[5] = cmul(w[4], w[1]); w[6] = cmul(w[4], w[2]); w[7] = cmul(w[4], w[3]);
        static_for<9, 16>([&](auto tc) { constexpr int tt = decltype(tc)::value; w[tt] = cmul(w[8], w[tt - 8]); });
        S[slot_of(q, 0)] = v[0];
        static_for<1, 16>([&](auto tc) { constexpr int tt = decltype(tc)::value; S[slot_of(q, tt)] = cmul_conj(v[tt], w[tt]); });
    }
}
// ------------------------------------------------------------------------------------------------ inverse, pass B
// `sink(jj, re, im)` receives real samples jj and jj + M (0 <= jj < M) of the inverse transform (unnormalised).
template <int N, class Sink>
TAC_HD void fft_inv_passB(int t, const cplx* __restrict__ S, Sink sink) {
    constexpr int M = N / 2, P = M / 16, CSTEP = 1024 / N;
    cplx v[P];
    static_for<0, P>([&](auto ic) { constexpr int i = decltype(ic)::value; v[i] = S[slot_of(bitrev<P>(i), t)]; });
    dft_inv<P>(v);
    static_for<0, P>([&](auto mc) {
        constexpr int m = decltype(mc)::value;
        const cplx z = mul_w128<false, m * CSTEP>(v[m]);
        sink(t + 16 * m, z.x, z.y);
    });
}

// `sink(mc, re, im)` with the register row m as a compile-time constant (samples t + 16m and t + 16m + M)
template <int N, class Sink>
TAC_HD void fft_inv_passB_m(int t, const cplx* __restrict__ S, Sink sink) {
    constexpr int M = N / 2, P = M / 16, CSTEP = 1024 / N;
    cplx v[P];
    static_for<0, P>([&](auto ic) { constexpr int i = decltype(ic)::value; v[i] = S[slot_of(bitrev<P>(i), t)]; });
    dft_inv<P>(v);
    static_for<0, P>([&](auto mc) {
        constexpr int m = decltype(mc)::value;
        const cplx z = mul_w128<false, m * CSTEP>(v[m]);
        sink(mc, z.x, z.y);
    });
}

// ------------------------------------------------------------------------------------------------ torus conversion
// fractional part of x (a real number whose integer part is irrelevant) as a torus element.
// [U] tfhe fft64/math/fft/mod.rs::convert_add_backward_torus
TAC_HD uint64_t f64_to_torus(double x) {
    const double C = 6755399441055744.0;     // 1.5 * 2^52: (x + C) - C == rint(x) for |x| < 2^51
    const double r = (x + C) - C;
    const double t = (x - r) * 18446744073709551616.0;
#if defined(__CUDA_ARCH__)
    return (uint64_t)__double2ll_rn(t);
#else
    if (t >= 9223372036854775808.0) return 1ull << 63;
    return (uint64_t)(int64_t)__builtin_nearbyint(t);
#endif
}
TAC_HD double torus_to_f64(uint64_t v) { return (double)(int64_t)v * (1.0 / 18446744073709551616.0); }

// ------------------------------------------------------------------------------------------------ decomposition for the f64 path
// All L signed digits of a torus value, bit-identical to tfhe's SignedDecomposer iterator (tac_common.h), computed once
// per coefficient and step.  Matching the iterator's tie rule matters even on the f64 path: a top-level tie resolved the
// other way yields a different (equally valid) ciphertext, which would make the ciphertext-level comparison of one
// external product with the oracle impossible.
// Digits are cached in shared memory as 16-bit fields  digit + B/2  (0 <= field <= B <= 2^15), the samples jj and jj + M
// packed in one 32-bit word — exactly the pair one FFT input register needs.
//
// Exact routine (all in 32-bit arithmetic, branch-free); returns the L fields packed 16 bits apiece, level 1 lowest:
//   y      = x + 2^(63-rep)                      rounding to the top rep = b·L bits
//   f_l    = bits [64-b·l, 64-b·(l-1)) of y      raw digit fields (f_1 is the most significant)
//   level l (from L down to 1):  r = f_l + carry_in;  carry_out = r > B/2  ||  (r == B/2 && tiebit_l);  digit = r - carry_out·B
//   tiebit_l = msb(f_{l-1}) for l > 1;  tiebit_1 = the iterator's "balance" decision
//            = f_1 > B/2 || (f_1 == B/2 && (lower fields != 0 || rounding bit))           (decomp_init_state)
// Equality with decomp_init_state/decomp_next, ties included, is checked in tests/test_ep_emulation.py.
template <int L>
TAC_HD uint64_t decompose_digits_exact(uint64_t x, int b) {
    static_assert(L <= 4, "packed result holds four 16-bit fields");
    const int rep = b * L;
    const uint32_t B = 1u << b, half = B >> 1, mask = B - 1u;
    const uint64_t y = x + (1ull << (63 - rep));
    const uint32_t rounding_bit = (uint32_t)(x >> (63 - rep)) & 1u;
    uint32_t f[L];
#pragma unroll
    for (int l = 1; l <= L; l++) f[l - 1] = (uint32_t)(y >> (64 - b * l)) & mask;
    uint32_t lower = 0;
#pragma unroll
    for (int l = 2; l <= L; l++) lower |= f[l - 1];
    const uint32_t balance = (f[0] > half) | ((f[0] == half) & ((lower != 0u) | rounding_bit));
    uint32_t carry = 0;
    uint64_t packed = 0;
#pragma unroll
    for (int l = L; l >= 1; l--) {
        const uint32_t r = f[l - 1] + carry;
        const uint32_t tiebit = (l > 1) ? (f[(l > 1) ? l - 2 : 0] >> (b - 1)) : balance;
        carry = (r > half) | ((r == half) & tiebit);
        packed |= (uint64_t)(r - (carry << b) + half) << (16 * (l - 1));
    }
    return packed;
}
// Fast path: the closed-form balanced decomposition
//     field_l = ((x + add) >> (64 - b·l)) & (B-1)  ( = digit_l + B/2 ),       add = rounding bit + B/2 at every level
// agrees with the iterator unless some level is an exact tie (raw digit == B/2  ⇔  field_l == 0, probability ≈ L·2^-b per
// coefficient); only then the exact routine above is replayed, out of line.  Everything stays in registers: the replay
// returns its fields by value.
struct DecompFast {
    uint64_t add;
    uint32_t mask;
    int b;
    double unbias;               // 2^52 + B/2: turns the magic-number conversion of a field into the signed digit
};
TAC_HD DecompFast make_decomp_fast(int b, int l) {
    DecompFast d;
    uint64_t add = 1ull << (63 - b * l);
    for (int lev = 1; lev <= l; lev++) add += (1ull << (b - 1)) << (64 - b * lev);
    d.add = add; d.mask = (1u << b) - 1u; d.b = b;
    d.unbias = 4503599627370496.0 + (double)(1u << (b - 1));
    return d;
}
#if defined(__CUDACC__)
template <int L> __device__ __noinline__ uint64_t decompose_digits_slow(uint64_t x, int b) { return decompose_digits_exact<L>(x, b); }
#else
template <int L> inline uint64_t decompose_digits_slow(uint64_t x, int b) { return decompose_digits_exact<L>(x, b); }
#endif
// fields of the samples x0 (low half-words) and x1 (high half-words), one word per level (lev-1 indexed)
template <int L>
TAC_HD void decompose_pair(uint64_t x0, uint64_t x1, const DecompFast& dc, uint32_t (&out)[L]) {
    const uint64_t y0 = x0 + dc.add, y1 = x1 + dc.add;
    uint32_t zero_probe = 0;
#pragma unroll
    for (int l = 1; l <= L; l++) {
        const uint32_t f0 = (uint32_t)(y0 >> (64 - dc.b * l)) & dc.mask;
        const uint32_t f1 = (uint32_t)(y1 >> (64 - dc.b * l)) & dc.mask;
        out[l - 1] = f0 | (f1 << 16);
        zero_probe |= out[l - 1] - 0x00010001u;           // bit 15 / 31 set iff a half-word was 0 (fields are < 2^15)
    }
    if (zero_probe & 0x80008000u) {                       // (a zero low half may also flag the high half: still a tie)
        const uint64_t p0 = decompose_digits_slow<L>(x0, dc.b), p1 = decompose_digits_slow<L>(x1, dc.b);
#pragma unroll
        for (int l = 1; l <= L; l++)
            out[l - 1] = ((uint32_t)(p0 >> (16 * (l - 1))) & 0xFFFFu) | (((uint32_t)(p1 >> (16 * (l - 1))) & 0xFFFFu) << 16);
    }
}
TAC_HD void unpack_digits(uint32_t w, const DecompFast& dc, double& a, double& b) {
    a = u32_magic(w & 0xFFFFu) - dc.unbias;
    b = u32_magic(w >> 16) - dc.unbias;
}
// coefficient j of (p · X^rot − p), rot in [0, 2N)
template <int N>
TAC_HD uint64_t rot_diff(const uint64_t* __restrict__ p, int j, int rot) {
    const int s = (j - rot) & (2 * N - 1);
    const uint64_t v = p[s & (N - 1)];
    constexpr int LOGN = (N == 256) ? 8 : (N == 512) ? 9 : (N == 1024) ? 10 : (N == 2048) ? 11 : -1;
    static_assert(LOGN > 0, "unsupported polynomial size");
    const uint64_t neg = (uint64_t)(s >> LOGN) & 1ull;
    return ((v ^ (0ull - neg)) + neg) - p[j];
}

// both coefficients jj and jj + N/2 of (p · X^rot − p) with the index arithmetic shared: adding N/2 to the rotated index
// flips bit log2(N)-1 and, when that bit was set, the sign
template <int N>
TAC_HD void rot_diff_pair(const uint64_t* __restrict__ p, int jj, int rot, uint64_t& x0, uint64_t& x1) {
    constexpr int LOGN = (N == 256) ? 8 : (N == 512) ? 9 : (N == 1024) ? 10 : (N == 2048) ? 11 : -1;
    static_assert(LOGN > 0, "unsupported polynomial size");
    const uint32_t s0 = (uint32_t)(jj - rot) & (uint32_t)(2 * N - 1);
    const uint32_t i0 = s0 & (uint32_t)(N - 1), i1 = i0 ^ (uint32_t)(N / 2);
    const uint32_t n0 = s0 >> LOGN, n1 = n0 ^ (i0 >> (LOGN - 1));
    const uint64_t v0 = p[i0], v1 = p[i1];
    const uint32_t m0 = 0u - n0, m1 = 0u - n1;
    const uint64_t w0 = ((uint64_t)((uint32_t)(v0 >> 32) ^ m0) << 32) | ((uint32_t)v0 ^ m0);
    const uint64_t w1 = ((uint64_t)((uint32_t)(v1 >> 32) ^ m1) << 32) | ((uint32_t)v1 ^ m1);
    x0 = (w0 + n0) - p[jj];
    x1 = (w1 + n1) - p[jj + N / 2];
}
}  // namespace tac
