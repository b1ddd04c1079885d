// tfhe_aes.hpp — C++ host mirror of the reference crate's layers L2–L4 for the B200 path (header only, sits on the C ABI).
//
//   namespace tfhe::cuda_woppbs_1bit   ↔  reference src/tfhe/shortint_woppbs_1bit.rs   (BitCt, FheContext, ClientKey, encode/decode)
//   namespace aes_128::fhe::data_model ↔  src/aes_128/fhe/data_model.rs                 (Byte, Word, Block, State, xor_state, shift_rows)
//   namespace aes_128::fhe::fhe_sbox_gal_mul_pbs ↔ src/aes_128/fhe/fhe_sbox_gal_mul_pbs.rs (generic AES over a ByteT policy)
//   namespace aes_128::fhe::fhe_impls  ↔  src/aes_128/fhe/fhe_impls/shortint_woppbs_1bit.rs:83-151 (LUT closures, Aes128Encrypt)
//
// Same names, argument meaning and error behaviour as the reference: Rust panics become exceptions with the same message
// ("noise components not independent", "NoiseTooBig", "cleartext out of bounds").  The generic AES code is written against
// a ByteT policy exactly like the reference's trait, so the per-byte path and the fused whole-round path are interchangeable.
#pragma once
#include "../../include/tfhe_aes_cuda.h"

#include <array>
#include <atomic>
#include <cstdint>
#include <algorithm>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

namespace tfhe {
namespace cuda_woppbs_1bit {

struct Panic : std::runtime_error { using std::runtime_error::runtime_error; };

inline uint64_t encode_bit(uint64_t bit) {                       // shortint_woppbs_1bit.rs:125-128
    if (bit >= 2) throw Panic("cleartext out of bounds: " + std::to_string(bit));
    return tac_encode_bit(bit);
}
inline uint64_t decode_bit(uint64_t encoding) { return tac_decode_bit(encoding); }   // :130-132

// :35-78
struct NoiseLevelWithComponents {
    uint64_t noise_level_squared = 0;
    std::set<uint64_t> components;
    static NoiseLevelWithComponents with_noise_level(uint64_t lvl, uint64_t id) { return {lvl, {id}}; }
    static NoiseLevelWithComponents trivial() { return {}; }
    void add_assign(const NoiseLevelWithComponents& rhs, uint64_t max_noise_level_squared) {
        for (uint64_t c : rhs.components)
            if (components.count(c)) throw Panic("noise components not independent");
        components.insert(rhs.components.begin(), rhs.components.end());
        noise_level_squared += rhs.noise_level_squared;
        if (noise_level_squared > max_noise_level_squared) throw Panic("NoiseTooBig");
    }
};

using LookupTable = std::pair<std::vector<uint64_t>, std::pair<int, int>>;   // table, (input_bits, output_bits)

// :166-172 — evaluation keys live in the HBM of one B200 behind the tac_ctx
class FheContext {
public:
    tac_params parameters{};
    FheContext(const tac_params& p, int device) : parameters(p), ctx_(tac_ctx_create(&p, device), tac_ctx_destroy) {
        if (!ctx_) throw Panic(std::string("tac_ctx_create failed: ") + tac_last_error(nullptr));
    }
    tac_ctx* raw() const { return ctx_.get(); }
    uint64_t next_ct_id() const { return ct_counter_->fetch_add(1); }                 // :175-178
    size_t lwe_size() const { return (size_t)parameters.glwe_dimension * parameters.polynomial_size + 1; }
    void check(int rc) const {
        if (rc == TAC_ERR_NOISE) throw Panic("NoiseTooBig");
        if (rc != TAC_OK) throw Panic(std::string("tfhe_aes_cuda: ") + tac_last_error(ctx_.get()));
    }
    // :274-289
    LookupTable generate_lookup_table(int input_bits, int output_bits, const std::function<uint64_t(uint16_t)>& f) const {
        std::vector<uint64_t> tab((size_t)1 << input_bits);
        for (size_t v = 0; v < tab.size(); v++) tab[v] = f((uint16_t)v);
        std::vector<uint64_t> lut(tac_lut_len(input_bits, parameters.polynomial_size) * (size_t)output_bits);
        if (tac_generate_lut(input_bits, output_bits, parameters.polynomial_size, tab.data(), lut.data()) != TAC_OK) throw Panic("generate_lookup_table: bad arguments");
        return {std::move(lut), {input_bits, output_bits}};
    }
    // the reference keeps one `static OnceLock` per LUT (fhe_impls/shortint_woppbs_1bit.rs:49,54,85,90,97) because it has one
    // parameter set per process; here a LUT belongs to the context that built it (another context may have another N)
    const LookupTable& cached_lut(int kind, int input_bits, int output_bits, const std::function<uint64_t(uint16_t)>& f) const {
        std::lock_guard<std::mutex> g(*mu_);
        auto it = named_luts_->find(kind);
        if (it == named_luts_->end()) it = named_luts_->emplace(kind, generate_lookup_table(input_bits, output_bits, f)).first;
        return it->second;
    }
    int lut_id(const LookupTable& lut) const {
        std::lock_guard<std::mutex> g(*mu_);
        auto it = lut_ids_->find(lut.first.data());
        if (it != lut_ids_->end()) return it->second;
        const int id = tac_lut_register(ctx_.get(), lut.second.first, lut.second.second, lut.first.data(), lut.first.size());
        if (id < 0) check(id);
        (*lut_ids_)[lut.first.data()] = id;
        return id;
    }
private:
    std::shared_ptr<tac_ctx> ctx_;
    std::shared_ptr<std::atomic<uint64_t>> ct_counter_ = std::make_shared<std::atomic<uint64_t>>(0);
    std::shared_ptr<std::mutex> mu_ = std::make_shared<std::mutex>();
    std::shared_ptr<std::map<const uint64_t*, int>> lut_ids_ = std::make_shared<std::map<const uint64_t*, int>>();
    std::shared_ptr<std::map<int, LookupTable>> named_luts_ = std::make_shared<std::map<int, LookupTable>>();
};

// :28-32, :86-122
struct BitCt {
    std::vector<uint64_t> ct;
    NoiseLevelWithComponents noise_level;
    const FheContext* context = nullptr;
    static BitCt with_noise_level(std::vector<uint64_t> ct, uint64_t lvl, const FheContext& c) {
        return {std::move(ct), NoiseLevelWithComponents::with_noise_level(lvl, c.next_ct_id()), &c};
    }
    static BitCt fresh(std::vector<uint64_t> ct, const FheContext& c) { return with_noise_level(std::move(ct), 1, c); }
    static BitCt trivial(uint64_t bit, const FheContext& c) {
        std::vector<uint64_t> ct(c.lwe_size(), 0);
        ct.back() = encode_bit(bit);
        return {std::move(ct), NoiseLevelWithComponents::trivial(), &c};
    }
    // BitXorAssign :134-142 (lwe_ciphertext_add_assign + bookkeeping)
    BitCt& operator^=(const BitCt& rhs) {
        noise_level.add_assign(rhs.noise_level, (uint64_t)context->parameters.max_noise_level_squared);
        for (size_t i = 0; i < ct.size(); i++) ct[i] += rhs.ct[i];
        return *this;
    }
    friend BitCt operator^(BitCt a, const BitCt& b) { a ^= b; return a; }
};

// FheContext::circuit_bootstrap :292-336 (and its batched form: `batch` independent calls, same LUT)
inline std::vector<std::vector<BitCt>> circuit_bootstrap_batch(const FheContext& ctx, const std::vector<std::vector<const BitCt*>>& calls, const LookupTable& lut) {
    const int n_in = lut.second.first, n_out = lut.second.second;
    const size_t L = ctx.lwe_size();
    std::vector<uint64_t> in(calls.size() * n_in * L), out(calls.size() * n_out * L);
    for (size_t q = 0; q < calls.size(); q++) {
        if ((int)calls[q].size() != n_in) throw Panic("circuit_bootstrap: wrong number of input bits");
        for (int i = 0; i < n_in; i++) std::copy(calls[q][i]->ct.begin(), calls[q][i]->ct.end(), in.begin() + (q * n_in + i) * L);
    }
    ctx.check(tac_wopbs_batch(ctx.raw(), ctx.lut_id(lut), (int)calls.size(), in.data(), out.data()));
    std::vector<std::vector<BitCt>> res(calls.size());
    for (size_t q = 0; q < calls.size(); q++)
        for (int o = 0; o < n_out; o++)
            res[q].push_back(BitCt::with_noise_level(std::vector<uint64_t>(out.begin() + (q * n_out + o) * L, out.begin() + (q * n_out + o + 1) * L),
                                                     (uint64_t)n_in /* NOMINAL × input_bit_count, :325 */, ctx));
    return res;
}
inline std::vector<BitCt> circuit_bootstrap(const FheContext& ctx, const std::vector<const BitCt*>& bits, const LookupTable& lut) {
    return circuit_bootstrap_batch(ctx, {bits}, lut)[0];
}

// :189-226
class ClientKey {
public:
    // seed == nullptr: 256 bits of OS entropy, like the reference (engine.rs:164-168); a seed gives reproducible — hence
    // publicly computable — keys and is for tests only
    ClientKey(const tac_params& p, const uint64_t* seed) : p_(p), ck_(seed ? tac_client_keygen(&p, *seed) : tac_client_keygen_os(&p), tac_client_free) {
        if (!ck_) throw Panic("client key generation failed (no OS entropy source)");
    }
    void gen_eval_keys(int threads = 0) { tac_client_gen_eval_keys(ck_.get(), threads); }
    void upload(const FheContext& ctx) {
        gen_eval_keys();
        ctx.check(tac_ctx_upload_keys(ctx.raw(), tac_client_key_ptr(ck_.get(), 2), tac_client_key_ptr(ck_.get(), 3), tac_client_key_ptr(ck_.get(), 4)));
    }
    BitCt encrypt(uint64_t bit, const FheContext& ctx) {                                   // ClientKeyT::encrypt
        if (bit >= 2) throw Panic("cleartext out of bounds: " + std::to_string(bit));
        std::vector<uint64_t> ct(ctx.lwe_size());
        const uint8_t b = (uint8_t)bit;
        tac_client_encrypt_bits(ck_.get(), &b, 1, counter_++, ct.data());
        return BitCt::fresh(std::move(ct), ctx);
    }
    uint64_t decrypt(const BitCt& bit) const {                                              // ClientKeyT::decrypt
        uint8_t b = 0;
        tac_client_decrypt_bits(ck_.get(), bit.ct.data(), 1, &b);
        return b;
    }
    tac_client_key* raw() const { return ck_.get(); }
private:
    tac_params p_;
    std::shared_ptr<tac_client_key> ck_;
    uint64_t counter_ = 0;
};

// FheContext::generate_keys_sqrd_lvl_{1,4,64,256} :229-243
inline std::pair<ClientKey, FheContext> generate_keys(int preset, const uint64_t* seed = nullptr, int device = 0) {
    tac_params p;
    if (tac_params_preset(preset, &p) != TAC_OK) throw Panic("unknown parameter preset");
    ClientKey ck(p, seed);
    FheContext ctx(p, device);
    ck.upload(ctx);
    return {std::move(ck), std::move(ctx)};
}

}  // namespace cuda_woppbs_1bit
}  // namespace tfhe

// ================================================================================================ AES
namespace aes_128 {

using Block = std::array<uint8_t, 16>;
using Key = std::array<uint8_t, 16>;
constexpr int ROUNDS = 10;
extern const uint8_t* const SBOX;          // 256 entries, generated in aes_plain.cpp
constexpr uint8_t RC[11] = {0x00, 0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40, 0x80, 0x1B, 0x36};
inline uint8_t gf_256_mul(uint8_t a, uint8_t b) {                // src/aes_128.rs:42-56
    uint8_t res = 0;
    for (int i = 0; i < 8; i++) {
        if (b & 1) res ^= a;
        const bool hi = a & 0x80;
        a = (uint8_t)(a << 1);
        if (hi) a ^= 0x1b;
        b >>= 1;
    }
    return res;
}

namespace plain {                                                // src/aes_128/plain.rs (clear AES with a `rounds` argument)
std::array<uint8_t, 176> key_schedule(const Key& key);
Block encrypt_block(const std::array<uint8_t, 176>& ek, const Block& block, int rounds);
}

namespace fhe {
namespace data_model {                                           // src/aes_128/fhe/data_model.rs
template <class Bit> using Byte = std::array<Bit, 8>;            // MSB first (:18-19)
template <class Bit> using Word = std::array<Byte<Bit>, 4>;      // :99-100
template <class Bit> using BlockT = std::array<Byte<Bit>, 16>;   // :165

template <class Bit, class Ctx> Byte<Bit> trivial_byte(const Ctx& ctx, uint8_t val) {      // Byte::trivial :35-43
    return {Bit::trivial((val >> 7) & 1, ctx), Bit::trivial((val >> 6) & 1, ctx), Bit::trivial((val >> 5) & 1, ctx), Bit::trivial((val >> 4) & 1, ctx),
            Bit::trivial((val >> 3) & 1, ctx), Bit::trivial((val >> 2) & 1, ctx), Bit::trivial((val >> 1) & 1, ctx), Bit::trivial(val & 1, ctx)};
}
template <class Bit> void xor_byte(Byte<Bit>& a, const Byte<Bit>& b) { for (int i = 0; i < 8; i++) a[i] ^= b[i]; }        // :73-78
template <class Bit> void xor_word(Word<Bit>& a, const Word<Bit>& b) { for (int i = 0; i < 4; i++) xor_byte(a[i], b[i]); }

// State of 4 rows each of 4 bytes (:169-188): state[row i][col j] = block[4j + i]
template <class Bit> struct State {
    std::array<Word<Bit>, 4> rows;
    static State from_array(BlockT<Bit> block) {
        State s;
        for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) s.rows[i][j] = std::move(block[4 * j + i]);
        return s;
    }
    BlockT<Bit> into_array() {
        BlockT<Bit> b;
        for (int i = 0; i < 16; i++) b[i] = std::move(rows[i % 4][i / 4]);
        return b;
    }
};
template <class Bit> void xor_state(State<Bit>& state, const Word<Bit>* key /* 4 words */) {   // AddRoundKey :270-274
    for (int j = 0; j < 4; j++) for (int i = 0; i < 4; i++) xor_byte(state.rows[i][j], key[j][i]);
}
template <class Bit> void shift_rows(State<Bit>& state) {                                     // :277-281 row i rotate_left(i)
    for (int i = 0; i < 4; i++) std::rotate(state.rows[i].begin(), state.rows[i].begin() + i, state.rows[i].end());
}
}  // namespace data_model

// src/aes_128/fhe/fhe_sbox_gal_mul_pbs.rs — generic over a ByteT policy (the reference's trait, :1-11):
//   static void bootstrap_assign(Byte&);  static Byte sbox_substitute(const Byte&);  static std::array<Byte,3> sbox_substitute_and_gal_mul(const Byte&);
// plus the batched hooks a device model may specialise (defaults call the per-byte functions).
namespace fhe_sbox_gal_mul_pbs {
using namespace data_model;

template <class Bit, class ByteT>
std::array<State<Bit>, 3> sub_bytes_with_gal_mul(State<Bit> state) {                          // :27-48
    auto bytes = state.into_array();
    auto muls = ByteT::sbox_substitute_and_gal_mul_all(bytes);                               // the reference's into_par_iter over 16 bytes
    std::array<BlockT<Bit>, 3> out;
    for (int b = 0; b < 16; b++) for (int m = 0; m < 3; m++) out[m][b] = std::move(muls[b][m]);
    return {State<Bit>::from_array(std::move(out[0])), State<Bit>::from_array(std::move(out[1])), State<Bit>::from_array(std::move(out[2]))};
}
template <class Bit>
State<Bit> mix_columns(std::array<State<Bit>, 3> m) {                                         // :61-82 (indices (i+3)%4, (i+2)%4, (i+1)%4: SURVEY §0.8)
    State<Bit> out;
    for (int j = 0; j < 4; j++)
        for (int i = 0; i < 4; i++) {
            Byte<Bit> b = m[1].rows[i][j];
            xor_byte(b, m[0].rows[(i + 3) % 4][j]);
            xor_byte(b, m[0].rows[(i + 2) % 4][j]);
            xor_byte(b, m[2].rows[(i + 1) % 4][j]);
            out.rows[i][j] = std::move(b);
        }
    return out;
}
template <class Bit, class ByteT>
BlockT<Bit> encrypt_block_for_rounds(const std::array<Word<Bit>, 44>& expanded_key, BlockT<Bit> block, int rounds) {   // :84-132
    auto state = State<Bit>::from_array(std::move(block));
    xor_state(state, &expanded_key[0]);
    for (int i = 1; i < rounds; i++) {
        auto muls = sub_bytes_with_gal_mul<Bit, ByteT>(std::move(state));
        for (auto& s : muls) shift_rows(s);
        state = mix_columns(std::move(muls));
        xor_state(state, &expanded_key[4 * i]);
    }
    auto bytes = state.into_array();                                                          // sub_bytes :51-58
    bytes = ByteT::sbox_substitute_all(bytes);
    state = State<Bit>::from_array(std::move(bytes));
    shift_rows(state);
    xor_state(state, &expanded_key[40]);                                                      // always round key 10 (:126-129)
    return state.into_array();
}
template <class Bit, class ByteT, class Ctx>
std::array<Word<Bit>, 44> key_schedule(const Ctx& ctx, const std::array<Byte<Bit>, 16>& key_slice) {                    // :134-164
    std::array<Word<Bit>, 44> ek;
    for (int i = 0; i < 4; i++) for (int j = 0; j < 4; j++) ek[i][j] = key_slice[4 * i + j];
    for (int i = 4; i < 44; i++) {
        if (i % 4 == 0) {
            Word<Bit> w = ek[i - 1];
            std::rotate(w.begin(), w.begin() + 1, w.end());                                   // rotate_left(1)
            for (auto& b : w) b = ByteT::sbox_substitute(b);                                  // sub_word :182-191
            ek[i] = ek[i - 4];
            xor_word(ek[i], w);
            xor_byte(ek[i][0], trivial_byte<Bit>(ctx, RC[i / 4]));
        } else {
            ek[i] = ek[i - 4];
            xor_word(ek[i], ek[i - 1]);
        }
        for (auto& b : ek[i]) ByteT::bootstrap_assign(b);                                     // boot_word :166-180
    }
    return ek;
}
}  // namespace fhe_sbox_gal_mul_pbs

// src/aes_128/fhe/fhe_impls/shortint_woppbs_1bit.rs:83-151 for the CUDA model
namespace fhe_impls {
namespace cuda_woppbs_1bit {
using tfhe::cuda_woppbs_1bit::BitCt;
using tfhe::cuda_woppbs_1bit::FheContext;
using tfhe::cuda_woppbs_1bit::LookupTable;
using Byte = data_model::Byte<BitCt>;

struct ByteT {
    static const FheContext& ctx_of(const Byte& b) { return *b[0].context; }
    static const LookupTable& identity_lut(const FheContext& c) { return c.cached_lut(0, 1, 1, [](uint16_t b) { return (uint64_t)b; }); }
    static const LookupTable& sbox_lut(const FheContext& c) { return c.cached_lut(1, 8, 8, [](uint16_t b) { return (uint64_t)SBOX[b]; }); }
    static const LookupTable& sbox_gal_mul_lut(const FheContext& c) {                                               // :97-111
        return c.cached_lut(2, 8, 24, [](uint16_t b) {
            return ((uint64_t)gf_256_mul(SBOX[b], 1) << 16) | ((uint64_t)gf_256_mul(SBOX[b], 2) << 8) | (uint64_t)gf_256_mul(SBOX[b], 3);
        });
    }
    static void bootstrap_assign(Byte& self) {                                                                      // :18-30 (8 one-bit boots, batched)
        const FheContext& c = ctx_of(self);
        std::vector<std::vector<const BitCt*>> calls;
        for (auto& bit : self) calls.push_back({&bit});
        auto out = tfhe::cuda_woppbs_1bit::circuit_bootstrap_batch(c, calls, identity_lut(c));
        for (int i = 0; i < 8; i++) self[i] = std::move(out[i][0]);
    }
    static Byte sbox_substitute(const Byte& self) { return sbox_substitute_all(std::array<Byte, 1>{self})[0]; }     // :32-44
    static std::array<Byte, 3> sbox_substitute_and_gal_mul(const Byte& self) { return sbox_substitute_and_gal_mul_all(std::array<Byte, 1>{self})[0]; }
    // the reference's rayon fan-out over the 16 bytes of a state becomes one batched call
    template <size_t NB> static std::array<Byte, NB> sbox_substitute_all(const std::array<Byte, NB>& bytes) {
        const FheContext& c = ctx_of(bytes[0]);
        std::vector<std::vector<const BitCt*>> calls(NB);
        for (size_t q = 0; q < NB; q++) for (auto& bit : bytes[q]) calls[q].push_back(&bit);
        auto out = tfhe::cuda_woppbs_1bit::circuit_bootstrap_batch(c, calls, sbox_lut(c));
        std::array<Byte, NB> res;
        for (size_t q = 0; q < NB; q++) for (int i = 0; i < 8; i++) res[q][i] = std::move(out[q][i]);
        return res;
    }
    template <size_t NB> static std::array<std::array<Byte, 3>, NB> sbox_substitute_and_gal_mul_all(const std::array<Byte, NB>& bytes) {   // :94-129
        const FheContext& c = ctx_of(bytes[0]);
        std::vector<std::vector<const BitCt*>> calls(NB);
        for (size_t q = 0; q < NB; q++) for (auto& bit : bytes[q]) calls[q].push_back(&bit);
        auto out = tfhe::cuda_woppbs_1bit::circuit_bootstrap_batch(c, calls, sbox_gal_mul_lut(c));
        std::array<std::array<Byte, 3>, NB> res;
        for (size_t q = 0; q < NB; q++) for (int m = 0; m < 3; m++) for (int i = 0; i < 8; i++) res[q][m][i] = std::move(out[q][m * 8 + i]);
        return res;
    }
};

// Aes128Encrypt (src/aes_128/fhe.rs:16-38) for the CUDA model: generic path (through ByteT) and fused device path
struct CudaWoppbs1BitSboxGalMulPbsAesEncrypt {
    using Ctx = FheContext;
    using Bit = BitCt;
    static data_model::BlockT<Bit> encrypt_block_for_rounds(const Ctx&, const std::array<data_model::Word<Bit>, 44>& ek, data_model::BlockT<Bit> block, int rounds) {
        return fhe_sbox_gal_mul_pbs::encrypt_block_for_rounds<Bit, ByteT>(ek, std::move(block), rounds);
    }
    static data_model::BlockT<Bit> encrypt_block(const Ctx& c, const std::array<data_model::Word<Bit>, 44>& ek, data_model::BlockT<Bit> block) {
        return encrypt_block_for_rounds(c, ek, std::move(block), ROUNDS);
    }
    static std::array<data_model::Word<Bit>, 44> key_schedule(const Ctx& c, const std::array<Byte, 16>& key) {
        return fhe_sbox_gal_mul_pbs::key_schedule<Bit, ByteT>(c, key);
    }
    // fused: all blocks × all rounds on the device (replaces main.rs:141-159's par_iter over blocks)
    static std::vector<data_model::BlockT<Bit>> encrypt_blocks_fused(const Ctx& c, const std::array<data_model::Word<Bit>, 44>& ek,
                                                                      const std::vector<data_model::BlockT<Bit>>& blocks, int rounds) {
        const size_t L = c.lwe_size();
        std::vector<uint64_t> ks(44 * 32 * L), in(blocks.size() * 128 * L), out(in.size());
        for (int w = 0; w < 44; w++) for (int b = 0; b < 4; b++) for (int i = 0; i < 8; i++) std::copy(ek[w][b][i].ct.begin(), ek[w][b][i].ct.end(), ks.begin() + ((w * 4 + b) * 8 + i) * L);
        uint64_t in_noise = 0;
        for (size_t q = 0; q < blocks.size(); q++) for (int b = 0; b < 16; b++) for (int i = 0; i < 8; i++) {
            std::copy(blocks[q][b][i].ct.begin(), blocks[q][b][i].ct.end(), in.begin() + ((q * 16 + b) * 8 + i) * L);
            in_noise = std::max(in_noise, blocks[q][b][i].noise_level.noise_level_squared);
        }
        c.check(tac_aes_set_key_schedule(c.raw(), ks.data()));
        c.check(tac_aes_encrypt_blocks(c.raw(), (int)blocks.size(), rounds, (int)in_noise, in.data(), out.data()));
        std::vector<data_model::BlockT<Bit>> res(blocks.size());
        for (size_t q = 0; q < blocks.size(); q++) for (int b = 0; b < 16; b++) for (int i = 0; i < 8; i++)
            res[q][b][i] = BitCt::with_noise_level(std::vector<uint64_t>(out.begin() + ((q * 16 + b) * 8 + i) * L, out.begin() + ((q * 16 + b) * 8 + i + 1) * L), 8 + 1, c);
        return res;
    }
    // AES over public blocks (AES-CTR counter blocks) under the device key schedule, no input ciphertexts; `xor` (empty or
    // one 16-byte row per block) is XORed into the output — the AES-CTR ciphertext for transciphering
    static std::vector<data_model::BlockT<Bit>> encrypt_public_blocks(const Ctx& c, const std::vector<std::array<uint8_t, 16>>& blocks, int rounds,
                                                                       const std::vector<std::array<uint8_t, 16>>& xor_bytes = {}) {
        return public_blocks(tac_aes_encrypt_public_blocks, c, blocks, rounds, xor_bytes);
    }
    // AES decryption (equivalent inverse cipher, FIPS-197 §5.3.5; the reference has none): derive the inverse key schedule
    // from the device key schedule, once per key schedule.  Decryption fails (TAC_ERR_STATE) until this has run.
    static void inv_key_schedule(const Ctx& c) { c.check(tac_aes_inv_key_schedule(c.raw(), nullptr)); }
    // decryption of public ciphertext blocks under the inverse key schedule; `xor` (empty or one 16-byte row per block) is
    // XORed into the output — the previous ciphertext blocks (IV first) for AES-CBC transciphering, empty for AES-ECB
    static std::vector<data_model::BlockT<Bit>> decrypt_public_blocks(const Ctx& c, const std::vector<std::array<uint8_t, 16>>& blocks, int rounds,
                                                                       const std::vector<std::array<uint8_t, 16>>& xor_bytes = {}) {
        return public_blocks(tac_aes_decrypt_public_blocks, c, blocks, rounds, xor_bytes);
    }

private:
    // fn (tac_aes_{en,de}crypt_public_blocks) over the blocks; outputs are bit ciphertexts of squared noise level 9
    static std::vector<data_model::BlockT<Bit>> public_blocks(int (*fn)(tac_ctx*, int, int, const uint8_t*, const uint8_t*, uint64_t*), const Ctx& c,
                                                              const std::vector<std::array<uint8_t, 16>>& blocks, int rounds,
                                                              const std::vector<std::array<uint8_t, 16>>& xor_bytes) {
        if (!xor_bytes.empty() && xor_bytes.size() != blocks.size()) throw std::invalid_argument("xor_bytes: one row per block");
        const size_t L = c.lwe_size();
        std::vector<uint64_t> out(blocks.size() * 128 * L);
        c.check(fn(c.raw(), (int)blocks.size(), rounds, blocks.empty() ? nullptr : blocks[0].data(), xor_bytes.empty() ? nullptr : xor_bytes[0].data(),
                   out.data()));
        std::vector<data_model::BlockT<Bit>> res(blocks.size());
        for (size_t q = 0; q < blocks.size(); q++) for (int b = 0; b < 16; b++) for (int i = 0; i < 8; i++)
            res[q][b][i] = BitCt::with_noise_level(std::vector<uint64_t>(out.begin() + ((q * 16 + b) * 8 + i) * L, out.begin() + ((q * 16 + b) * 8 + i + 1) * L), 8 + 1, c);
        return res;
    }
};
}  // namespace cuda_woppbs_1bit
}  // namespace fhe_impls

// src/aes_128/fhe/fhe_encryption.rs
namespace fhe_encryption {
using tfhe::cuda_woppbs_1bit::BitCt;
using tfhe::cuda_woppbs_1bit::ClientKey;
using tfhe::cuda_woppbs_1bit::FheContext;
inline data_model::Byte<BitCt> encrypt_byte(ClientKey& ck, const FheContext& c, uint8_t byte) {
    data_model::Byte<BitCt> b;
    for (int i = 0; i < 8; i++) b[i] = ck.encrypt((byte >> (7 - i)) & 1, c);               // util::u8_to_bits, MSB first
    return b;
}
template <size_t N> std::array<data_model::Byte<BitCt>, N> encrypt_byte_array(ClientKey& ck, const FheContext& c, const std::array<uint8_t, N>& a) {
    std::array<data_model::Byte<BitCt>, N> r;
    for (size_t i = 0; i < N; i++) r[i] = encrypt_byte(ck, c, a[i]);
    return r;
}
inline uint8_t decrypt_byte(const ClientKey& ck, const data_model::Byte<BitCt>& b) {
    uint8_t v = 0;
    for (int i = 0; i < 8; i++) v |= (uint8_t)(ck.decrypt(b[i]) << (7 - i));
    return v;
}
template <size_t N> std::array<uint8_t, N> decrypt_byte_array(const ClientKey& ck, const std::array<data_model::Byte<BitCt>, N>& a) {
    std::array<uint8_t, N> r;
    for (size_t i = 0; i < N; i++) r[i] = decrypt_byte(ck, a[i]);
    return r;
}
}  // namespace fhe_encryption
}  // namespace fhe
}  // namespace aes_128
