// aes_gcm.cpp — AES-GCM formatting (SP 800-38D §7.2, 96-bit IVs), GF(2^128) in GCM's bit order, the linear-layer planner
// (aes_gcm.h) and the host-only C export tac_aes_gcm_format.
#include "aes_gcm.h"

#include <algorithm>
#include <cstring>
#include <map>

namespace tac {

Gf128 gf128_from_block(const uint8_t b[16]) {
    Gf128 x;
    for (int i = 0; i < 128; i++)
        if (b[i >> 3] & (0x80 >> (i & 7))) x.flip(i);
    return x;
}
void gf128_to_block(const Gf128& x, uint8_t b[16]) {
    std::memset(b, 0, 16);
    for (int i = 0; i < 128; i++)
        if (x.bit(i)) b[i >> 3] |= (uint8_t)(0x80 >> (i & 7));
}
Gf128 gf128_mul_x(const Gf128& x) {
    const bool carry = (x.hi >> 63) != 0;
    Gf128 r{x.lo << 1, (x.hi << 1) | (x.lo >> 63)};
    if (carry) r.lo ^= 0x87;                 // x^128 = x^7 + x^2 + x + 1
    return r;
}
Gf128 gf128_mul(const Gf128& a, const Gf128& b) {
    Gf128 r, s = b;
    for (int i = 0; i < 128; i++) {
        if (a.bit(i)) { r.lo ^= s.lo; r.hi ^= s.hi; }
        s = gf128_mul_x(s);
    }
    return r;
}
std::vector<int> gf128_fold(int u) {
    Gf128 x;
    x.flip(std::min(u, 127));
    for (int k = 127; k < u; k++) x = gf128_mul_x(x);
    std::vector<int> out;
    for (int i = 0; i < 128; i++)
        if (x.bit(i)) out.push_back(i);
    return out;
}

uint64_t gf128_box_fn(int v) {
    uint64_t prod = 0;                       // bit t: coefficient t
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++)
            if (((v >> (7 - i)) & 1) && ((v >> (3 - j)) & 1)) prod ^= 1ull << (i + j);
    uint64_t f = 0;                          // output t is bit 6 − t of f
    for (int t = 0; t < 7; t++)
        if ((prod >> t) & 1) f |= 1ull << (6 - t);
    return f;
}

void gf128_rows(int np, std::vector<LinRow>& rows) {
    rows.assign((size_t)np * 128, LinRow{});
    std::vector<std::vector<int>> fold(255);
    for (int u = 0; u < 255; u++) fold[u] = gf128_fold(u);
    for (int p = 0; p < np; p++)
        for (int i = 0; i < 32; i++)
            for (int j = 0; j < 32; j++)
                for (int t = 0; t < 7; t++) {
                    const int u = 4 * (i + j) + t;
                    const uint64_t row = ((uint64_t)p * 1024 + i * 32 + j) * 7 + t;
                    for (int r : fold[u]) rows[(size_t)p * 128 + r].terms.push_back(LinTerm{lin_id(0, row), 8, (int64_t)p * 256 + u});
                }
}

int gcm_shape(const tac_ccm_msg& msg, GcmShape& s) {
    if (msg.nonce_len != 12 || !msg.nonce) return TAC_ERR_ARG;
    if (!(msg.tag_len == 4 || msg.tag_len == 8 || (msg.tag_len >= 12 && msg.tag_len <= 16))) return TAC_ERR_ARG;
    if (msg.data_len < (uint64_t)msg.tag_len || (msg.data_len > 0 && !msg.data) || (msg.aad_len > 0 && !msg.aad)) return TAC_ERR_ARG;
    s.t = msg.tag_len;
    s.p = msg.data_len - (uint64_t)msg.tag_len;
    if (s.p > (1ull << 36) - 32 || msg.aad_len >= (1ull << 61)) return TAC_ERR_ARG;       // SP 800-38D §5.2.1.1
    s.m = (int64_t)((s.p + 15) / 16);
    s.aad_blocks = (int64_t)((msg.aad_len + 15) / 16);
    s.M = s.aad_blocks + s.m + 1;
    return TAC_OK;
}

void gcm_ctr_block(const tac_ccm_msg& msg, uint32_t i, uint8_t out[16]) {
    std::memcpy(out, msg.nonce, 12);
    for (int k = 0; k < 4; k++) out[12 + k] = (uint8_t)(i >> (24 - 8 * k));
}

void gcm_ghash_blocks(const tac_ccm_msg& msg, const GcmShape& s, uint8_t* out) {
    std::memset(out, 0, (size_t)s.M * 16);
    if (msg.aad_len) std::memcpy(out, msg.aad, (size_t)msg.aad_len);
    if (s.p) std::memcpy(out + 16 * s.aad_blocks, msg.data, (size_t)s.p);
    uint8_t* len = out + 16 * (s.M - 1);
    const uint64_t bits[2] = {8 * (uint64_t)msg.aad_len, 8 * s.p};
    for (int h = 0; h < 2; h++)
        for (int k = 0; k < 8; k++) len[8 * h + k] = (uint8_t)(bits[h] >> (56 - 8 * k));
}

void ghash_terms(const uint8_t* blocks, int n, const int* exps, int src, uint64_t base, int64_t seg0, LinRow* rows) {
    for (int i = 0; i < n; i++) {
        Gf128 col = gf128_from_block(blocks + 16 * (size_t)i);          // X_i · x^l, l = 0, 1, …
        const uint64_t r0 = base + 128 * (uint64_t)(exps[i] - 1);
        for (int l = 0; l < 128; l++) {
            for (int j = 0; j < 128; j++)
                if (col.bit(j)) rows[j].terms.push_back(LinTerm{lin_id(src, r0 + l), 1, seg0 + i});
            col = gf128_mul_x(col);
        }
    }
}

int lin_plan_build(const std::vector<LinRow>& rows_in, int max_noise, int out_limit, int first_src, LinPlan& plan) {
    plan = LinPlan{};
    std::vector<std::vector<LinTerm>> rows(rows_in.size());
    for (size_t r = 0; r < rows.size(); r++) {
        rows[r] = rows_in[r].terms;
        for (const LinTerm& t : rows[r])
            if (t.nu > max_noise) return TAC_ERR_ARG;
    }
    auto noise = [](const std::vector<LinTerm>& ts) {
        int64_t s = 0;
        for (const LinTerm& t : ts) s += t.nu;
        return s;
    };
    for (int level = 0;; level++) {
        bool any = false;
        for (auto& ts : rows) any |= noise(ts) > out_limit;
        if (!any) break;
        const int src = first_src + level;
        if (src >= kLinMaxSrc) return TAC_ERR_ARG;
        LinSums lv;
        std::map<std::vector<uint32_t>, uint32_t> index;        // a group's sorted term ids → its row in this level
        auto refresh = [&](const std::vector<LinTerm>& g) {
            std::vector<uint32_t> key;
            for (const LinTerm& t : g) key.push_back(t.id);
            std::sort(key.begin(), key.end());
            auto it = index.find(key);
            if (it == index.end()) {
                it = index.emplace(key, (uint32_t)lv.rows()).first;
                for (const LinTerm& t : g) lv.terms.push_back(t.id);
                lv.row_ptr.push_back((uint32_t)lv.terms.size());
            }
            return LinTerm{lin_id(src, it->second), 1, -(((int64_t)level + 1) << 40) - (int64_t)it->second};
        };
        for (auto& ts : rows) {
            const int64_t s = noise(ts);
            if (s <= out_limit) continue;
            std::vector<LinTerm> next;
            if (s <= max_noise) {
                next.push_back(refresh(ts));
            } else {
                // segments in order of first appearance, each cut into runs that fit; single terms are packed together
                std::vector<int64_t> segs;
                std::map<int64_t, std::vector<LinTerm>> by_seg;
                for (const LinTerm& t : ts) {
                    auto& v = by_seg[t.seg];
                    if (v.empty()) segs.push_back(t.seg);
                    v.push_back(t);
                }
                std::vector<LinTerm> singles;
                for (int64_t sg : segs) {
                    std::vector<LinTerm> cur;
                    int64_t cn = 0;
                    auto close = [&]() {
                        if (cur.size() == 1) singles.push_back(cur[0]);
                        else if (!cur.empty()) next.push_back(refresh(cur));
                        cur.clear(); cn = 0;
                    };
                    for (const LinTerm& t : by_seg[sg]) {
                        if (cn + t.nu > max_noise) close();
                        cur.push_back(t); cn += t.nu;
                    }
                    close();
                }
                const bool progress = !next.empty();
                std::vector<LinTerm> cur;
                int64_t cn = 0;
                auto close = [&]() {
                    if (cur.size() > 1 || (cur.size() == 1 && !progress && cur[0].nu > 1)) next.push_back(refresh(cur));
                    else if (cur.size() == 1) next.push_back(cur[0]);
                    cur.clear(); cn = 0;
                };
                for (const LinTerm& t : singles) {
                    if (cn + t.nu > max_noise) close();
                    cur.push_back(t); cn += t.nu;
                }
                close();
            }
            ts.swap(next);
        }
        plan.levels.push_back(std::move(lv));
    }
    for (size_t r = 0; r < rows.size(); r++) {
        for (const LinTerm& t : rows[r]) plan.final.terms.push_back(t.id);
        plan.final.row_ptr.push_back((uint32_t)plan.final.terms.size());
        plan.final.cbit.push_back(rows_in[r].cbit);
    }
    return TAC_OK;
}

}  // namespace tac

extern "C" int tac_aes_gcm_format(const tac_ccm_msg* msg, uint8_t* ctr_blocks, uint8_t* ghash_blocks, int64_t counts[2]) {
    tac::GcmShape s;
    if (!msg || !counts) return TAC_ERR_ARG;
    if (int rc = tac::gcm_shape(*msg, s)) return rc;
    counts[0] = s.m + 1;
    counts[1] = s.M;
    if (ctr_blocks)
        for (int64_t i = 0; i <= s.m; i++) tac::gcm_ctr_block(*msg, (uint32_t)(i + 1), ctr_blocks + 16 * i);
    if (ghash_blocks) tac::gcm_ghash_blocks(*msg, s, ghash_blocks);
    return TAC_OK;
}
