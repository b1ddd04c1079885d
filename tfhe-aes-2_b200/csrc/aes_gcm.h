// aes_gcm.h — host side of AES-GCM transciphering (NIST SP 800-38D, 96-bit IVs): formatting of the counter blocks and the
// GHASH blocks, GF(2^128) in GCM's bit order, and the planner of the linear layer (aes_gcm.cpp).  Pure integer, no device.
//
// Bit order: coefficient i of a block is bit i counted MSB first (byte i/8, bit 7 − i%8), which is row 8·byte + bit of the
// device layout [16][8][kN+1].  GHASH_H(X_1..X_M) = Σ_i X_i · H^(M+1−i).
//
// The linear layer: "output row j = XOR of these terms, term t carrying squared noise ν_t, plus a public constant bit".
// A sum whose noise exceeds max_noise_level_squared cannot be bootstrapped, so the planner builds levels: each level forms
// group sums that fit the budget and refreshes them with a 1-bit circuit bootstrap (squared noise 1 afterwards), until
// every row's sum fits the consumer's limit; a final gather-add then writes the rows.  Groups never mix terms of different
// segments unless a segment's terms stand alone, and groups with equal terms are formed once, so rows that share a
// segment (the partial products of one unreduced coefficient in a GF(2^128) product) share its refreshes.
#pragma once
#include <cstdint>
#include <vector>

#include "../../include/tfhe_aes_cuda.h"

namespace tac {

// ---------------------------------------------------------------------------------------------- GF(2^128), GCM order
// bit i of the pair (lo: coefficients 0..63, hi: 64..127) is the coefficient of x^i
struct Gf128 {
    uint64_t lo = 0, hi = 0;
    bool bit(int i) const { return ((i < 64 ? lo >> i : hi >> (i - 64)) & 1) != 0; }
    void flip(int i) { if (i < 64) lo ^= 1ull << i; else hi ^= 1ull << (i - 64); }
};
Gf128 gf128_from_block(const uint8_t b[16]);
void gf128_to_block(const Gf128& x, uint8_t b[16]);
Gf128 gf128_mul_x(const Gf128& x);                        // x · X mod x^128 + x^7 + x^2 + x + 1
Gf128 gf128_mul(const Gf128& a, const Gf128& b);
// x^u reduced, for u < 255: the output coefficients an unreduced product coefficient u folds into
std::vector<int> gf128_fold(int u);

// ---------------------------------------------------------------------------------------------- records
// the shape of one record: p payload bytes, m = ceil(p/16) counter blocks after J0, M GHASH blocks (AAD, C, lengths)
struct GcmShape {
    int t = 0;
    uint64_t p = 0;
    int64_t m = 0, aad_blocks = 0, M = 0;
};
// checks one record (IV of 12 bytes, tag length in {4, 8, 12, 13, 14, 15, 16}, data_len >= tag_len, p <= 2^36 − 32,
// aad_len < 2^61, no NULL pointer with a non-zero length) and gives its shape; TAC_OK or TAC_ERR_ARG
int gcm_shape(const tac_ccm_msg& msg, GcmShape& s);
void gcm_ctr_block(const tac_ccm_msg& msg, uint32_t i, uint8_t out[16]);         // IV ‖ BE32(i): J0 is i = 1
void gcm_ghash_blocks(const tac_ccm_msg& msg, const GcmShape& s, uint8_t* out);  // [M][16]: AAD, C (zero-padded), lengths

// ---------------------------------------------------------------------------------------------- the linear layer
// a term reads row `row` of source `src` (device array src of a gather-add); sources 0..7
constexpr int kLinSrcShift = 29;
inline uint32_t lin_id(int src, uint64_t row) { return ((uint32_t)src << kLinSrcShift) | (uint32_t)row; }
constexpr uint64_t kLinMaxRow = 1ull << kLinSrcShift;
constexpr int kLinMaxSrc = 8;

struct LinTerm {
    uint32_t id;
    int nu;            // squared noise
    int64_t seg;       // segment
};
struct LinRow {
    std::vector<LinTerm> terms;
    uint8_t cbit = 0;  // public constant bit XORed in
};
// one gather-add: out row r = Σ terms[row_ptr[r] .. row_ptr[r+1]) (+ 2^63 on the body when cbit[r])
struct LinSums {
    std::vector<uint32_t> row_ptr{0}, terms;
    std::vector<uint8_t> cbit;
    size_t rows() const { return row_ptr.size() - 1; }
};
// levels[k]: group sums, refreshed; their outputs are source first_src + k.  final: the rows as asked.
struct LinPlan {
    std::vector<LinSums> levels;
    LinSums final;
    size_t refreshes() const {
        size_t n = 0;
        for (const LinSums& l : levels) n += l.rows();
        return n;
    }
};
// plans rows so that every output row has squared noise <= out_limit (or 1 when refreshed) and no bootstrap input exceeds
// max_noise; sources first_src and up are the levels'.  TAC_ERR_ARG when a term exceeds max_noise, or the levels need
// more than kLinMaxSrc sources.
int lin_plan_build(const std::vector<LinRow>& rows, int max_noise, int out_limit, int first_src, LinPlan& plan);

// the 8 → 7 box of the product: inputs a_0..a_3, b_0..b_3 (coefficients, input 0 the LUT's MSB), output t = coefficient
// t of the carry-less product (output 0 the LUT's MSB); f for tac_generate_lut
uint64_t gf128_box_fn(int v);

// the sums of np products: output bit r of product p = XOR of the box outputs (p, i, j, t) (row ((p·1024 + 32i + j)·7 + t)
// of source 0, squared noise 8) whose unreduced coefficient u = 4(i + j) + t folds into r; segment (p, u), so the groups of
// one u serve every r it folds into
void gf128_rows(int np, std::vector<LinRow>& rows);

// Σ_i X_i · H^(e_i) over the n blocks X_i [n][16] as terms of a power table (source src, H^e bit l at row
// base + 128·(e − 1) + l, squared noise 1): row j gains H^(e_i) bit l for every l with bit j of X_i · x^l; block i is
// segment seg0 + i
void ghash_terms(const uint8_t* blocks, int n, const int* exps, int src, uint64_t base, int64_t seg0, LinRow* rows /* [128] */);

}  // namespace tac
