// aes_plan.h — which circuit bootstraps of AES over PUBLIC blocks are equal across blocks (aes_plan.cpp).
//
// State byte j (= 4·col + row) entering the S-box of round r depends on the input bytes D(r, j):
//   D(1, j) = {j},   D(r+1, (row, c)) = ∪_{r'=0..3} D(r, 4·((c + r') mod 4) + r')        (ShiftRows + MixColumns)
// and on nothing else but the (shared) key schedule.  So in round r, byte j of blocks a and b bootstraps the same
// ciphertext exactly when a and b agree on every byte of D(r, j).  Round 1 shares per byte value, round 2 per
// diagonal, and from round 3 on D covers all 16 bytes: only identical blocks share.
//
// The equivalent inverse cipher (tac_aes_decrypt_public_blocks) spreads dependence along the other diagonal:
//   D(r+1, (row, c)) = ∪_{r'=0..3} D(r, 4·((c − r') mod 4) + r')                             (InvShiftRows + InvMixColumns)
//
// Under many keys (a per-block key index into a table of key schedules) the key schedule is shared only among blocks of
// the same key: two positions share a bootstrap when their blocks have the same key index AND agree on D(r, j).
#pragma once
#include <cstdint>
#include <vector>

namespace tac {

struct AesRoundPlan {
    int64_t boxes = 0;               // representatives = circuit bootstraps this round
    bool identity = false;           // boxes == 16·n: representative k is position k (block k/16, byte k%16)
    std::vector<int32_t> rep_pos;    // [boxes]    position block·16 + byte of each representative (its first occurrence)
    std::vector<int32_t> idx;        // [n·16]     representative of every position
};

enum class AesDir { Forward, Inverse };

// plan[r-1] for r = 1..rounds of the cipher in direction `dir`; key_idx: NULL (one key) or the key index of every block.
// Returns TAC_OK or TAC_ERR_ARG (n_blocks < 0, rounds outside 1..10, NULL blocks with n_blocks > 0, a negative key index)
int aes_public_plan_build(int n_blocks, int rounds, const uint8_t* blocks /*[n][16]*/, AesDir dir, std::vector<AesRoundPlan>& plan,
                          const int32_t* key_idx = nullptr /*[n]*/);

}  // namespace tac
