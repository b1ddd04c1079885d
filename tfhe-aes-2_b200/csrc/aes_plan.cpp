// aes_plan.cpp — the sharing plan of AES over public blocks (aes_plan.h) and its C exports tac_aes_public_plan[_inv].
// Host only, pure integer: the CPU tests pin it down, and tac_aes_{en,de}crypt_public_blocks[_dev] run exactly this plan.
#include "aes_plan.h"
#include "../../include/tfhe_aes_cuda.h"

#include <algorithm>
#include <string>
#include <unordered_map>

namespace tac {

int aes_public_plan_build(int n_blocks, int rounds, const uint8_t* blocks, AesDir dir, std::vector<AesRoundPlan>& plan) {
    if (n_blocks < 0 || rounds < 1 || rounds > 10 || (n_blocks > 0 && !blocks)) return TAC_ERR_ARG;
    plan.assign(rounds, AesRoundPlan{});
    const size_t npos = (size_t)n_blocks * 16;
    const int sgn = dir == AesDir::Forward ? 1 : -1;        // (c ± r') mod 4: ShiftRows or InvShiftRows
    uint16_t dep[16];                                       // D(r, j) as a bit mask over the 16 input bytes
    for (int j = 0; j < 16; j++) dep[j] = (uint16_t)(1u << j);
    for (int r = 1; r <= rounds; r++) {
        if (r > 1) {
            uint16_t next[16];
            for (int j = 0; j < 16; j++) {
                const int c = j >> 2;
                next[j] = 0;
                for (int rr = 0; rr < 4; rr++) next[j] |= dep[4 * ((c + sgn * rr) & 3) + rr];
            }
            std::copy(next, next + 16, dep);
        }
        AesRoundPlan& p = plan[r - 1];
        p.idx.resize(npos);
        // one table per byte position: the bytes of D(r, j) (others zeroed) → representative
        std::vector<std::unordered_map<std::string, int32_t>> seen(16);
        for (auto& m : seen) m.reserve((size_t)n_blocks);
        std::string key(16, '\0');
        for (int b = 0; b < n_blocks; b++)
            for (int j = 0; j < 16; j++) {
                for (int i = 0; i < 16; i++) key[i] = (dep[j] >> i & 1) ? (char)blocks[(size_t)b * 16 + i] : '\0';
                const int32_t pos = b * 16 + j;
                auto ins = seen[j].emplace(key, (int32_t)p.rep_pos.size());
                if (ins.second) p.rep_pos.push_back(pos);
                p.idx[pos] = ins.first->second;
            }
        p.boxes = (int64_t)p.rep_pos.size();
        // representatives are numbered in order of first occurrence, so 16·n of them means rep k sits at position k
        p.identity = (size_t)p.boxes == npos;
    }
    return TAC_OK;
}

}  // namespace tac

static int export_plan(int n_blocks, int rounds, const uint8_t* blocks_host, tac::AesDir dir, int64_t* boxes) {
    std::vector<tac::AesRoundPlan> plan;
    if (int rc = tac::aes_public_plan_build(n_blocks, rounds, blocks_host, dir, plan)) return rc;
    if (!boxes) return TAC_ERR_ARG;
    for (int r = 0; r < rounds; r++) boxes[r] = plan[r].boxes;
    return TAC_OK;
}
extern "C" int tac_aes_public_plan(int n_blocks, int rounds, const uint8_t* blocks_host, int64_t* boxes) {
    return export_plan(n_blocks, rounds, blocks_host, tac::AesDir::Forward, boxes);
}
extern "C" int tac_aes_public_plan_inv(int n_blocks, int rounds, const uint8_t* blocks_host, int64_t* boxes) {
    return export_plan(n_blocks, rounds, blocks_host, tac::AesDir::Inverse, boxes);
}
