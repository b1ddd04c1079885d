// kernels_common.cuh — the integer / glue kernels of the WoP-PBS hot path (SURVEY.md §8a rows a3, a12 fallback, a17).
// The FFT / external-product kernels live in kernels_ep.cuh, the tensor-core keyswitch GEMMs in kernels_gemm_umma.cuh.
//
//   pfks_digits_kernel     digits of the private functional packing keyswitch for the integer-pipe GEMM (base_log > 16)
//   lwe_gemm_kernel        exact integer GEMM mod 2^64 on the integer pipe: out[ct][col] = corr[col] − Σ_k digit'[ct][k]·key[k][col]
//                          (PFKS of params_sqrd_lvl_1, and the correction rows of both keyswitches at key upload)
//   aes_*_kernel           AddRoundKey / (Inv)ShiftRows+(Inv)MixColumns+AddRoundKey / final round as gather-adds on the flat
//                          state (aes_mix_columns_kernel and aes_final_round_kernel templated on the direction); round-1
//                          inputs and representative gathers of the public-block path; InvMixColumns of the inverse key
//                          schedule (aes_inv_mix_key_kernel); the sums of a batched key-expansion step (aes_key_step_kernel)
//   aes_ccm_*_kernel       AES-CCM: the CBC-MAC chain input X ⊕ B of one step, and the tag difference the tag check bootstraps
//   lwe_gather_add_kernel  the linear layer of AES-GCM (aes_gcm.h): rows as sums of rows of several arrays, plus a constant bit
//   lwe_add_kernel         leveled XOR (lwe_ciphertext_add_assign) over a batch; lwe_shl_kernel / lwe_sub_kernel: glue of extract_bits
//   negate_kernel, dfma_peak_kernel   key-upload helper, FP64 peak microbenchmark (roofline denominator)
#pragma once
#include <cuda_runtime.h>
#include "tac_common.h"
#include "aes_ccm.h"

namespace tac {


// ================================================================================================ digits
// bit-exact signed decomposition (tfhe SignedDecomposer), stored with the offset B/2 so that digits are non-negative:
// digit' = digit + B/2 ∈ [0, B].
// PFKS: closest_representable first, all big+1 elements (mask and body), key block stores level 1 first and is iterated
// reversed ([U] lwe_private_functional_packing_keyswitch.rs).
__global__ void pfks_digits_kernel(const uint64_t* __restrict__ in, int nct, int big1, int b, int l, uint32_t* __restrict__ dig) {
    const size_t total = (size_t)nct * big1;
    for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
        uint64_t st = decomp_init_state(closest_representable(in[idx], b, l), b, l);
        uint32_t* o = dig + idx * l;
        for (int lev = l; lev >= 1; lev--) o[lev - 1] = (uint32_t)(decomp_next(st, b) + (int64_t)(1u << (b - 1)));
    }
}

// ================================================================================================ integer GEMM mod 2^64
// out[ct][j][col] = corr[j][col] − Σ_k dig[ct][k] · key[j][k][col]   (+ last_col_add[ct·stride] on col == W-1)
// CTA tile: (4·RB ciphertexts) × 128 columns; thread: RB ciphertexts × 2 adjacent columns; K chunked by 32 through smem.
// The product u32 × u64 → low 64 bits is one IMAD.WIDE.U32 (low limb, 64-bit accumulate) plus one IMAD (high limb).
template <int RB>
__global__ void __launch_bounds__(256)
lwe_gemm_kernel(const uint32_t* __restrict__ dig, int nct, int Kd, const uint64_t* __restrict__ key, int W, int nkeys,
                const uint64_t* __restrict__ corr, const uint64_t* __restrict__ last_col_add, size_t add_stride,
                uint64_t* __restrict__ out) {
    constexpr int TB = 4 * RB, KC = 32, TN = 128;
    __shared__ __align__(16) uint32_t dsm[TB][KC];
    const int tiles_per_key = (W + TN - 1) / TN;
    const int j = blockIdx.x / tiles_per_key;
    const int col = (blockIdx.x - j * tiles_per_key) * TN + 2 * (threadIdx.x & 63);
    const int ty = threadIdx.x >> 6;
    const int ct0 = blockIdx.y * TB;
    const bool col_ok = col < W;           // W is even, so col+1 < W as well
    uint64_t acc[RB][2];
#pragma unroll
    for (int r = 0; r < RB; r++) { acc[r][0] = 0; acc[r][1] = 0; }
    const uint64_t* kbase = key + (size_t)j * Kd * W + (col_ok ? col : 0);
    for (int k0 = 0; k0 < Kd; k0 += KC) {
        for (int e = threadIdx.x; e < TB * KC; e += 256) {
            const int r = e / KC, kk = e - r * KC;
            const int ct = ct0 + r, k = k0 + kk;
            dsm[r][kk] = (ct < nct && k < Kd) ? dig[(size_t)ct * Kd + k] : 0u;
        }
        __syncthreads();
        const int kmax = min(KC, Kd - k0);
        if (col_ok) {
#pragma unroll 4
            for (int kk = 0; kk < kmax; kk++) {
                const ulonglong2 kv = __ldg(reinterpret_cast<const ulonglong2*>(kbase + (size_t)(k0 + kk) * W));
                const uint32_t k0lo = (uint32_t)kv.x, k0hi = (uint32_t)(kv.x >> 32), k1lo = (uint32_t)kv.y, k1hi = (uint32_t)(kv.y >> 32);
#pragma unroll
                for (int r = 0; r < RB; r++) {
                    const uint32_t d = dsm[ty * RB + r][kk];
                    acc[r][0] += (uint64_t)d * k0lo; acc[r][0] += (uint64_t)(d * k0hi) << 32;
                    acc[r][1] += (uint64_t)d * k1lo; acc[r][1] += (uint64_t)(d * k1hi) << 32;
                }
            }
        }
        __syncthreads();
    }
    if (!col_ok) return;
    const uint64_t c0 = corr ? corr[(size_t)j * W + col] : 0ull, c1 = corr ? corr[(size_t)j * W + col + 1] : 0ull;
#pragma unroll
    for (int r = 0; r < RB; r++) {
        const int ct = ct0 + ty * RB + r;
        if (ct >= nct) continue;
        uint64_t v0 = c0 - acc[r][0], v1 = c1 - acc[r][1];
        if (last_col_add && col + 1 == W - 1) v1 += last_col_add[(size_t)ct * add_stride];   // W is even: the last column is a v1
        uint64_t* o = out + ((size_t)ct * nkeys + j) * W + col;
        *reinterpret_cast<ulonglong2*>(o) = make_ulonglong2(v0, v1);
    }
}

// ================================================================================================ AES linear layers
// flat state: [block][byte = 4·col + row][bit, MSB first][L]   (reference data_model.rs:165-188 re-expressed)
// Round keys of block b: rk, or rk + kidx[b]·key_words when a per-block key index is given (AES under many keys: rk points
// into entry 0 of a table of key schedules `key_words` apart).
__device__ __forceinline__ const uint64_t* aes_block_key(const uint64_t* rk, const int32_t* kidx, size_t key_words, size_t blk) {
    return kidx ? rk + (size_t)kidx[blk] * key_words : rk;
}
// AddRoundKey (data_model.rs:270-274): out = in + rk, rk broadcast over blocks
__global__ void aes_add_round_key_kernel(const uint64_t* __restrict__ in, const uint64_t* __restrict__ rk, size_t blk_words, size_t total,
                                         uint64_t* __restrict__ out, const int32_t* __restrict__ kidx, size_t key_words) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t blk = i / blk_words;
        out[i] = in[i] + aes_block_key(rk, kidx, key_words, blk)[i - blk * blk_words];
    }
}
// ShiftRows + MixColumns + AddRoundKey of a middle round as one gather-add over the S-box rows; Fwd = false is InvShiftRows +
// InvMixColumns of the equivalent inverse cipher (FIPS-197 §5.3.5, round keys from dk):
//   new[row][c] = Σ_rr coef[(rr − row) mod 4] · S(old[rr][(c ± rr) mod 4])       (+ for ShiftRows, − for InvShiftRows)
//   forward  coef = {2, 3, 1, 1}      muls rows [24 = (S, 2S, 3S) × 8 bits][L]               (fhe_sbox_gal_mul_pbs.rs:61-82, :106-117)
//   inverse  coef = {14, 11, 13, 9}   muls rows [32 = (14, 11, 13, 9)·InvS × 8 bits][L]
// row = block·16 + byte, or idx[block·16 + byte] when idx is given (a compact batch of S-box outputs shared by several
// positions: AES over public blocks); round keys per block as in aes_add_round_key_kernel
template <bool Fwd>
__global__ void aes_mix_columns_kernel(const uint64_t* __restrict__ muls, const uint64_t* __restrict__ rk, int L, size_t total,
                                       uint64_t* __restrict__ state, const int32_t* __restrict__ idx, const int32_t* __restrict__ kidx,
                                       size_t key_words) {
    constexpr int W = Fwd ? 24 : 32;
    const size_t byte_words = (size_t)8 * L, blk_words = 16 * byte_words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t blk = i / blk_words; const size_t rem = i - blk * blk_words;
        const int byte = (int)(rem / byte_words); const size_t w = rem - (size_t)byte * byte_words;   // bit·L + e
        const int c = byte >> 2, r = byte & 3;
        uint64_t v = aes_block_key(rk, kidx, key_words, blk)[rem];
#pragma unroll
        for (int rr = 0; rr < 4; rr++) {
            const int d = (rr - r) & 3;
            const int slot = Fwd ? (d < 2 ? d + 1 : 0) : d;                  // muls slot of coef[d]
            const int old_byte = 4 * ((Fwd ? c + rr : c - rr) & 3) + rr;
            const size_t src_row = idx ? (size_t)idx[blk * 16 + old_byte] : blk * 16 + old_byte;
            v += muls[(src_row * W + (size_t)slot * 8) * L + w];
        }
        state[i] = v;
    }
}
// last round (fhe_sbox_gal_mul_pbs.rs:119-129): ShiftRows(S) + w[40..43], or InvShiftRows(InvS) + dk[0..3].  sub rows
// [row][8 bits][L] (idx optional, as in aes_mix_columns_kernel).  xr: NULL, or [block][16] public bytes XORed into the
// output (a trivial ciphertext added: encode_bit(1) = 2^63 on the body of every set bit).  Round keys per block as in
// aes_add_round_key_kernel.
template <bool Fwd>
__global__ void aes_final_round_kernel(const uint64_t* __restrict__ sub, const uint64_t* __restrict__ rk, int L, size_t total,
                                       uint64_t* __restrict__ out, const int32_t* __restrict__ idx,
                                       const uint8_t* __restrict__ xr, const int32_t* __restrict__ kidx, size_t key_words) {
    const size_t byte_words = (size_t)8 * L, blk_words = 16 * byte_words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t blk = i / blk_words; const size_t rem = i - blk * blk_words;
        const int byte = (int)(rem / byte_words); const size_t w = rem - (size_t)byte * byte_words;
        const int c = byte >> 2, r = byte & 3;
        const int old_byte = 4 * ((Fwd ? c + r : c - r) & 3) + r;
        const size_t src_row = idx ? (size_t)idx[blk * 16 + old_byte] : blk * 16 + old_byte;
        uint64_t v = sub[src_row * byte_words + w] + aes_block_key(rk, kidx, key_words, blk)[rem];
        if (xr) {
            const int bit = (int)(w / L);
            if (w - (size_t)bit * L == (size_t)L - 1 && (xr[blk * 16 + byte] & (0x80 >> bit))) v += 1ull << 63;
        }
        out[i] = v;
    }
}
// S-box inputs of round 1 over public blocks, one per representative k: k0[byte] + trivial(value), i.e. the key-schedule
// byte with encode_bit(1) = 2^63 added to the body of every set bit of the public byte (Byte::trivial, data_model.rs:35-43).
// rep_pos[k] = block·16 + byte (NULL: k itself); out [k][8 bits][L].  The key is the one of the representative's block
// (kidx as in aes_add_round_key_kernel; positions that share a representative share its key, aes_plan.h).
__global__ void aes_public_round1_kernel(const uint64_t* __restrict__ k0, const uint8_t* __restrict__ blocks, const int32_t* __restrict__ rep_pos,
                                         int L, size_t total, uint64_t* __restrict__ out, const int32_t* __restrict__ kidx, size_t key_words) {
    const size_t byte_words = (size_t)8 * L;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t k = i / byte_words; const size_t w = i - k * byte_words;
        const int pos = rep_pos ? rep_pos[k] : (int)k;
        const int bit = (int)(w / L);
        uint64_t v = aes_block_key(k0, kidx, key_words, (size_t)(pos >> 4))[(size_t)(pos & 15) * byte_words + w];
        if (w - (size_t)bit * L == (size_t)L - 1 && (blocks[pos] & (0x80 >> bit))) v += 1ull << 63;
        out[i] = v;
    }
}
// inverse key schedule, dk[4rd..4rd+3] = InvMixColumns(w[4rd..4rd+3]): InvMixColumns without the shift over round keys.
// muls: [key byte][32 = (14, 11, 13, 9)·b × 8 bits][L] for consecutive round keys of 16 bytes; out [key byte][8 bits][L]
// (squared noise 4·8 = 32, bootstrapped back to level 1 by the caller)
__global__ void aes_inv_mix_key_kernel(const uint64_t* __restrict__ muls, int L, size_t total, uint64_t* __restrict__ out) {
    const size_t byte_words = (size_t)8 * L, blk_words = 16 * byte_words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t blk = i / blk_words; const size_t rem = i - blk * blk_words;
        const int byte = (int)(rem / byte_words); const size_t w = rem - (size_t)byte * byte_words;
        const int c = byte >> 2, r = byte & 3;
        uint64_t v = 0;
#pragma unroll
        for (int rr = 0; rr < 4; rr++) v += muls[((blk * 16 + 4 * c + rr) * 32 + (size_t)((rr - r) & 3) * 8) * L + w];
        out[i] = v;
    }
}
// one step i (4 <= i < 44) of the key expansion over K schedules ek [K][44 words][4 bytes][8 bits][L] (sched_words apart):
//   acc[k] = w[i−4] + RotWord(sub[k]) + trivial(RC)   when sub is given (i % 4 == 0: sub[k] = SubWord(w[i−1]), unrotated)
//   acc[k] = w[i−4] + w[i−1]                          otherwise
// rc: the 8 ciphertexts of trivial(RC[i/4]) added to byte 0; acc [K][4][8][L], bootstrapped back to level 1 by the caller
__global__ void aes_key_step_kernel(const uint64_t* __restrict__ ek, size_t sched_words, int i, const uint64_t* __restrict__ sub,
                                    const uint64_t* __restrict__ rc, int L, size_t total, uint64_t* __restrict__ acc) {
    const size_t byte_words = (size_t)8 * L, word = 4 * byte_words;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
        const size_t k = t / word; const size_t w = t - k * word;
        const uint64_t* e = ek + k * sched_words;
        uint64_t v = e[(size_t)(i - 4) * word + w];
        if (sub) {
            const int byte = (int)(w / byte_words);
            v += sub[k * word + (size_t)((byte + 1) & 3) * byte_words + (w - (size_t)byte * byte_words)];   // rotate_left(1): bytes [1,2,3,0]
            if (byte == 0) v += rc[w];
        } else {
            v += e[(size_t)(i - 1) * word + w];
        }
        acc[t] = v;
    }
}
// the representatives' S-box inputs out of the full state: out[k] = state[rep_pos[k]], 8·L words each
__global__ void aes_gather_bytes_kernel(const uint64_t* __restrict__ state, const int32_t* __restrict__ rep_pos, int L, size_t total,
                                        uint64_t* __restrict__ out) {
    const size_t byte_words = (size_t)8 * L;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t k = i / byte_words; const size_t w = i - k * byte_words;
        out[i] = state[(size_t)rep_pos[k] * byte_words + w];
    }
}
// ================================================================================================ AES-CCM (aes_ccm.h)
// CBC-MAC chain input of one step over the first a active messages (sorted order): out[j] = X[j] ⊕ B, where X[j] is row j
// of the public call's output `pub` (the chain state, updated in place by the caller) and B is, by desc[j] (CcmChainDesc),
// the first len bytes of the FHE plaintext row desc[j].src of `pub` (zero padding: nothing added) or the public AAD bytes
// as a trivial ciphertext (encode_bit(1) = 2^63 on the body of every set bit, as xr in aes_final_round_kernel).
// total = a·16·8·L words.
__global__ void aes_ccm_chain_input_kernel(const uint64_t* __restrict__ pub, const CcmChainDesc* __restrict__ desc, int L, size_t total,
                                           uint64_t* __restrict__ out) {
    const size_t byte_words = (size_t)8 * L, blk_words = 16 * byte_words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t j = i / blk_words; const size_t rem = i - j * blk_words;
        const int byte = (int)(rem / byte_words); const size_t w = rem - (size_t)byte * byte_words;
        const CcmChainDesc& d = desc[j];
        uint64_t v = pub[i];
        if (d.src >= 0) {
            if (byte < d.len) v += pub[(size_t)d.src * blk_words + rem];
        } else {
            const int bit = (int)(w / L);
            if (w - (size_t)bit * L == (size_t)L - 1 && (d.aad[byte] & (0x80 >> bit))) v += 1ull << 63;
        }
        out[i] = v;
    }
}
// tag difference, message c in the caller's order: D[c][b] = X[r][b] ⊕ (E(A_0) ⊕ U)[r][b] for bytes b < tag_len[c], trivial
// zero for the rest, r = rank[c] its sorted row.  X = rows 0..n−1 of `pub`, E(A_0) ⊕ U = rows n..2n−1.  D is zero exactly
// when the tag is genuine.  out [n][16][8][L]; total = n·16·8·L words.
__global__ void aes_ccm_tag_diff_kernel(const uint64_t* __restrict__ pub, const int32_t* __restrict__ rank, const int32_t* __restrict__ tag_len,
                                        int n, int L, size_t total, uint64_t* __restrict__ out) {
    const size_t byte_words = (size_t)8 * L, blk_words = 16 * byte_words;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t c = i / blk_words; const size_t rem = i - c * blk_words;
        const int byte = (int)(rem / byte_words);
        const size_t r = (size_t)rank[c];
        out[i] = byte < tag_len[c] ? pub[r * blk_words + rem] + pub[((size_t)n + r) * blk_words + rem] : 0ull;
    }
}

// ================================================================================================ linear layer (aes_gcm.h)
// the gather-add's inputs: any device ciphertext arrays [rows][L], addressed by a term's source (its top 3 bits).  The
// output may lie in one of them when no row reads what another writes (out is not __restrict__).
struct LinSrcs {
    const uint64_t* p[8];
};
// out row r (at out_row[r] when given) = Σ_{t in [row_ptr[r], row_ptr[r+1])} row (terms[t] & 2^29−1) of source terms[t] >> 29,
// mod 2^64, + 2^63 on the body when cbit[r] (a public constant bit: a trivial ciphertext).  A row without terms is a
// trivial zero.  total = rows·L words.
__global__ void lwe_gather_add_kernel(LinSrcs src, const uint32_t* __restrict__ row_ptr, const uint32_t* __restrict__ terms,
                                      const uint8_t* __restrict__ cbit, const uint32_t* __restrict__ out_row, int L, size_t total,
                                      uint64_t* out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / L; const size_t e = i - r * L;
        uint64_t v = 0;
        for (uint32_t t = row_ptr[r], end = row_ptr[r + 1]; t < end; t++) {
            const uint32_t id = __ldg(terms + t), k = id >> 29;
            const uint64_t* base = src.p[0];
#pragma unroll
            for (uint32_t q = 1; q < 8; q++) base = k == q ? src.p[q] : base;      // selects: an indexed parameter would go to the stack
            v += base[(size_t)(id & ((1u << 29) - 1)) * L + e];
        }
        if (cbit && cbit[r] && e == (size_t)L - 1) v += 1ull << 63;
        out[(out_row ? (size_t)out_row[r] : r) * L + e] = v;
    }
}

// leveled XOR (BitXorAssign, shortint_woppbs_1bit.rs:134-142 → lwe_ciphertext_add_assign): a += b, element-wise
__global__ void lwe_add_kernel(uint64_t* __restrict__ a, const uint64_t* __restrict__ b, size_t total) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) a[i] += b[i];
}
// bit extraction glue ([U] wop_pbs.rs::extract_bits): out = a · 2^shift, a −= b
__global__ void lwe_shl_kernel(const uint64_t* __restrict__ a, int shift, size_t total, uint64_t* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) out[i] = a[i] << shift;
}
__global__ void lwe_sub_kernel(uint64_t* __restrict__ a, const uint64_t* __restrict__ b, size_t total) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) a[i] -= b[i];
}
__global__ void negate_kernel(uint64_t* __restrict__ a, size_t total) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) a[i] = 0ull - a[i];
}

// FP64 FMA throughput probe: 16 independent DFMA chains per thread
__global__ void dfma_peak_kernel(double* __restrict__ sink, int iters, double m) {
    double a[16];
#pragma unroll
    for (int i = 0; i < 16; i++) a[i] = 1.0 + 1e-9 * (threadIdx.x + i);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int i = 0; i < 16; i++) a[i] = fma(a[i], m, 1e-12);
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) s += a[i];
    if (s == 123.456) sink[0] = s;
}

}  // namespace tac
