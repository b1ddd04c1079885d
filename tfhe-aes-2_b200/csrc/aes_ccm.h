// aes_ccm.h — host side of AES-CCM transciphering (NIST SP 800-38C, RFC 3610): formatting of B_0, the AAD blocks and the
// counter blocks, and the schedule of one batched call (aes_ccm.cpp).  Pure integer, no device.
//
// One call over n messages runs
//   1. one public-block AES call over [B_0 of every message][A_0 of every message][A_1..A_m of every message], with XOR
//      bytes 0, U ‖ 0…, and C zero-padded: rows 0..n−1 are X_1 = E(B_0), rows n..2n−1 are E(A_0) ⊕ U (the expected tag
//      when it is genuine), the rest is the FHE plaintext;
//   2. the CBC-MAC chain X_{s+1} = E(X_s ⊕ B_s) on the encrypted-block path, in place on rows 0..n−1.  Messages are
//      sorted by chain length, descending, so the messages that still have a block s are a prefix of a_s rows;
//   3. the tag check on MSB_t(X_final) ⊕ E(A_0) ⊕ U.
// All rows are in sorted message order; `order` maps back to the caller's.
#pragma once
#include <cstdint>
#include <vector>

#include "../../include/tfhe_aes_cuda.h"

namespace tac {

// chain input of one active message in one step: src >= 0 is the public-call row of its FHE plaintext block, of which the
// first len bytes are valid (zero padding adds nothing); src < 0 means the block is public AAD bytes, added as a trivial
// ciphertext.  Uploaded as is to the device (aes_ccm_chain_input_kernel).
struct CcmChainDesc {
    int32_t src;
    int32_t len;
    uint8_t aad[16];
};

// the shape of one message: q = 15 − |N|, p = payload bytes, m payload blocks, aad_blocks AAD blocks with the length prefix
struct CcmShape {
    int q = 0, t = 0;
    uint64_t p = 0;
    int64_t m = 0, aad_blocks = 0;
    int64_t chain() const { return aad_blocks + m; }    // CBC-MAC steps after X_1 = E(B_0)
};

// checks one message (nonce length 7..13, tag length in {4, 6, …, 16}, data_len >= tag_len, p < 2^(8q), no NULL pointer
// with a non-zero length) and gives its shape; TAC_OK or TAC_ERR_ARG
int ccm_shape(const tac_ccm_msg& msg, CcmShape& s);

// B_0 (16 bytes), the AAD blocks (16·aad_blocks bytes, length prefix and zero padding included) and A_i (16 bytes)
void ccm_b0(const tac_ccm_msg& msg, const CcmShape& s, uint8_t* out);
void ccm_aad_blocks(const tac_ccm_msg& msg, const CcmShape& s, uint8_t* out);
void ccm_ctr_block(const tac_ccm_msg& msg, const CcmShape& s, uint64_t i, uint8_t* out);

// the schedule of one batched call over n messages (validated by the caller)
struct CcmPlan {
    int n = 0;
    std::vector<CcmShape> shape;          // [n] caller order
    std::vector<int32_t> order;           // [n] sorted position → caller index (chain length descending, stable)
    std::vector<int32_t> rank;            // [n] caller index → sorted position
    std::vector<int64_t> pt_row;          // [n] caller order: public-call row of A_1 (its first p bytes are the plaintext)
    std::vector<int64_t> pt_off;          // [n] caller order: first plaintext byte in the output [Σ p][8][kN+1]
    uint64_t pt_bytes = 0;                // Σ p
    // the public call: [2n + Σ m] blocks, XOR bytes and (keyed) per-row key index
    std::vector<uint8_t> pub_blocks, pub_xor;
    std::vector<int32_t> pub_kidx;        // empty without a key index
    std::vector<int32_t> kidx_sorted;     // [n] key index in sorted order (empty without one)
    // the chain: step s = 1..steps runs over the first active[s−1] sorted messages; desc holds active[s−1] entries per step
    std::vector<int32_t> active;
    std::vector<uint8_t> adds_plaintext;  // [steps] 1 when some active message adds an FHE plaintext block (squared noise 18)
    std::vector<CcmChainDesc> desc;
    std::vector<int32_t> tag_len;         // [n] caller order
};

// builds the plan; key_idx NULL (one schedule) or one index per message (range checked by the caller)
void ccm_plan_build(int n, const tac_ccm_msg* msgs, const int32_t* key_idx, CcmPlan& plan);

}  // namespace tac
