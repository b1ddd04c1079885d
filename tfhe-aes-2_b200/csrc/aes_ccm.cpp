// aes_ccm.cpp — AES-CCM formatting (SP 800-38C Appendix A) and the schedule of a batched transciphering call (aes_ccm.h),
// and the host-only C export tac_aes_ccm_format.  The CPU tests replay this formatting in clear AES against a reference
// AES-CCM, and tac_aes_ccm_transcipher[_dev] run exactly this plan.
#include "aes_ccm.h"

#include <algorithm>
#include <cstring>

namespace tac {

int ccm_shape(const tac_ccm_msg& msg, CcmShape& s) {
    if (msg.nonce_len < 7 || msg.nonce_len > 13 || !msg.nonce) return TAC_ERR_ARG;
    if (msg.tag_len < 4 || msg.tag_len > 16 || (msg.tag_len & 1)) return TAC_ERR_ARG;
    if (msg.data_len < (uint64_t)msg.tag_len || (msg.data_len > 0 && !msg.data) || (msg.aad_len > 0 && !msg.aad)) return TAC_ERR_ARG;
    // lengths far beyond any record (and beyond what fits the block counts below)
    if (msg.data_len >> 60 || msg.aad_len >> 60) return TAC_ERR_ARG;
    s.q = 15 - msg.nonce_len;
    s.t = msg.tag_len;
    s.p = msg.data_len - (uint64_t)msg.tag_len;
    if (s.q < 8 && (s.p >> (8 * s.q)) != 0) return TAC_ERR_ARG;         // [p]_q must hold p
    s.m = (int64_t)((s.p + 15) / 16);
    if (msg.aad_len == 0) {
        s.aad_blocks = 0;
    } else {
        const uint64_t prefix = msg.aad_len < 0xFF00u ? 2 : (msg.aad_len >> 32) == 0 ? 6 : 10;
        s.aad_blocks = (int64_t)((prefix + msg.aad_len + 15) / 16);
    }
    return TAC_OK;
}

static void put_be(uint64_t v, int len, uint8_t* out) {
    for (int i = len - 1; i >= 0; i--, v >>= 8) out[i] = (uint8_t)(v & 0xFF);
}

void ccm_b0(const tac_ccm_msg& msg, const CcmShape& s, uint8_t* out) {
    out[0] = (uint8_t)((msg.aad_len > 0 ? 64 : 0) + 8 * ((s.t - 2) / 2) + (s.q - 1));
    std::memcpy(out + 1, msg.nonce, (size_t)msg.nonce_len);
    put_be(s.p, s.q, out + 16 - s.q);
}

void ccm_aad_blocks(const tac_ccm_msg& msg, const CcmShape& s, uint8_t* out) {
    const size_t total = (size_t)s.aad_blocks * 16;
    if (total == 0) return;
    std::memset(out, 0, total);
    size_t off;
    if (msg.aad_len < 0xFF00u) {
        put_be(msg.aad_len, 2, out); off = 2;
    } else if ((msg.aad_len >> 32) == 0) {
        out[0] = 0xFF; out[1] = 0xFE; put_be(msg.aad_len, 4, out + 2); off = 6;
    } else {
        out[0] = 0xFF; out[1] = 0xFF; put_be(msg.aad_len, 8, out + 2); off = 10;
    }
    std::memcpy(out + off, msg.aad, (size_t)msg.aad_len);
}

void ccm_ctr_block(const tac_ccm_msg& msg, const CcmShape& s, uint64_t i, uint8_t* out) {
    out[0] = (uint8_t)(s.q - 1);
    std::memcpy(out + 1, msg.nonce, (size_t)msg.nonce_len);
    put_be(i, s.q, out + 16 - s.q);
}

void ccm_plan_build(int n, const tac_ccm_msg* msgs, const int32_t* key_idx, CcmPlan& plan) {
    plan = CcmPlan{};
    plan.n = n;
    plan.shape.resize(n);
    for (int c = 0; c < n; c++) ccm_shape(msgs[c], plan.shape[c]);
    plan.order.resize(n);
    for (int c = 0; c < n; c++) plan.order[c] = c;
    std::stable_sort(plan.order.begin(), plan.order.end(), [&](int32_t a, int32_t b) { return plan.shape[a].chain() > plan.shape[b].chain(); });
    plan.rank.resize(n);
    for (int r = 0; r < n; r++) plan.rank[plan.order[r]] = r;

    // the public call: [B_0 rows][A_0 rows][A_1..A_m rows], sorted order
    int64_t rows = 2 * (int64_t)n;
    plan.pt_row.resize(n);
    for (int r = 0; r < n; r++) {
        const int c = plan.order[r];
        plan.pt_row[c] = rows;
        rows += plan.shape[c].m;
    }
    plan.pt_off.resize(n);
    plan.tag_len.resize(n);
    for (int c = 0; c < n; c++) {
        plan.pt_off[c] = (int64_t)plan.pt_bytes;
        plan.pt_bytes += plan.shape[c].p;
        plan.tag_len[c] = plan.shape[c].t;
    }
    plan.pub_blocks.assign((size_t)rows * 16, 0);
    plan.pub_xor.assign((size_t)rows * 16, 0);
    if (key_idx) {
        plan.pub_kidx.resize((size_t)rows);
        plan.kidx_sorted.resize(n);
    }
    for (int r = 0; r < n; r++) {
        const int c = plan.order[r];
        const tac_ccm_msg& msg = msgs[c];
        const CcmShape& s = plan.shape[c];
        ccm_b0(msg, s, &plan.pub_blocks[(size_t)r * 16]);
        ccm_ctr_block(msg, s, 0, &plan.pub_blocks[(size_t)(n + r) * 16]);
        std::memcpy(&plan.pub_xor[(size_t)(n + r) * 16], msg.data + s.p, (size_t)s.t);                  // U ‖ 0…
        for (int64_t i = 1; i <= s.m; i++) ccm_ctr_block(msg, s, (uint64_t)i, &plan.pub_blocks[(size_t)(plan.pt_row[c] + i - 1) * 16]);
        if (s.p) std::memcpy(&plan.pub_xor[(size_t)plan.pt_row[c] * 16], msg.data, (size_t)s.p);          // C, zero-padded
        if (key_idx) {
            plan.kidx_sorted[r] = key_idx[c];
            plan.pub_kidx[r] = plan.pub_kidx[n + r] = key_idx[c];
            for (int64_t i = 0; i < s.m; i++) plan.pub_kidx[(size_t)(plan.pt_row[c] + i)] = key_idx[c];
        }
    }

    // the chain: sorted by length, so the messages with a block s are the first active[s−1]
    const int64_t steps = n ? plan.shape[plan.order[0]].chain() : 0;
    std::vector<std::vector<uint8_t>> aad(n);
    for (int c = 0; c < n; c++) {
        aad[c].resize((size_t)plan.shape[c].aad_blocks * 16);
        ccm_aad_blocks(msgs[c], plan.shape[c], aad[c].data());
    }
    int a = n;
    for (int64_t s = 1; s <= steps; s++) {
        while (a > 0 && plan.shape[plan.order[a - 1]].chain() < s) a--;
        plan.active.push_back(a);
        uint8_t adds = 0;
        for (int j = 0; j < a; j++) {
            const int c = plan.order[j];
            const CcmShape& sh = plan.shape[c];
            CcmChainDesc d{};
            if (s <= sh.aad_blocks) {
                d.src = -1;
                std::memcpy(d.aad, &aad[c][(size_t)(s - 1) * 16], 16);
            } else {
                const int64_t i = s - sh.aad_blocks;                     // payload block i = 1..m
                d.src = (int32_t)(plan.pt_row[c] + i - 1);
                d.len = (int32_t)std::min<uint64_t>(16, sh.p - 16 * (uint64_t)(i - 1));
                adds = 1;
            }
            plan.desc.push_back(d);
        }
        plan.adds_plaintext.push_back(adds);
    }
}

}  // namespace tac

extern "C" int tac_aes_ccm_format(const tac_ccm_msg* msg, uint8_t* ctr_blocks, uint8_t* mac_blocks, int64_t counts[2]) {
    tac::CcmShape s;
    if (!msg || !counts) return TAC_ERR_ARG;
    if (int rc = tac::ccm_shape(*msg, s)) return rc;
    counts[0] = s.m + 1;
    counts[1] = s.chain() + 1;
    if (ctr_blocks)
        for (int64_t i = 0; i <= s.m; i++) tac::ccm_ctr_block(*msg, s, (uint64_t)i, ctr_blocks + 16 * i);
    if (mac_blocks) {
        tac::ccm_b0(*msg, s, mac_blocks);
        tac::ccm_aad_blocks(*msg, s, mac_blocks + 16);
        std::memset(mac_blocks + 16 * (1 + s.aad_blocks), 0, (size_t)s.m * 16);
    }
    return TAC_OK;
}
