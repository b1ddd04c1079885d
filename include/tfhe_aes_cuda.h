/* tfhe_aes_cuda.h — C ABI of the B200 implementation of tfhe-aes-2's WoP-PBS hot path.
 *
 * The reference (allanbrondum/tfhe-aes-2) has no FFI: its boundary is the Rust trait set of SURVEY.md §8(b).  Every
 * entry point below names the reference item it replaces (file:line under the reference's src/).  A Rust `-sys` crate binds
 * these 1:1 (INTEGRATION.md shows the stubs); this repo's own host mirrors (Python ctypes in tfhe-aes-2_b200/__init__.py,
 * C++ in tfhe-aes-2_b200/host/) sit on exactly the same symbols.
 *
 * Conventions
 *   - every function returns 0 on success, a negative tac_status otherwise; tac_last_error() gives the message.  The
 *     reference panics on these conditions (assert!/unwrap), so a binding turns non-zero into a panic.
 *   - all buffers are caller-owned, little-endian uint64 torus words (q = 2^64).  `_dev` variants take device pointers
 *     and enqueue on the context's stream without synchronising; the plain variants take HOST pointers, copy in, run,
 *     copy out and synchronise.
 *   - LWE ciphertext   = mask[dim] ‖ body                      (big key: dim = k·N; small key: dim = n)
 *     GLWE ciphertext  = k mask polynomials ‖ body polynomial, N coefficients each
 *     GGSW (standard)  = [level s (decomposition level s+1)][row r = 0..k][poly c = 0..k][N]
 *     BSK  (standard)  = [i = 0..n-1] GGSW(s_i)                                 (pbs_level, pbs_base_log)
 *     KSK              = [i = 0..kN-1][s = 0..l-1 (decomposition level l-s)][n+1] (ks_level, ks_base_log)
 *     PFPKSK           = [j = 0..k][i = 0..kN (last = body)][s (level s+1)][(k+1)N] (pfks_level, pfks_base_log)
 *     LUT              = [n_out][N << max(0, n_in − log2 N)]     (reference WopbsLUTBase)
 *     AES block        = [16 bytes][8 bits, MSB first][kN+1];  key schedule = [44 words][4 bytes][8 bits][kN+1]
 *   - thread safety: every entry point may be called concurrently from any number of host threads on the same tac_ctx
 *     (the reference calls circuit_bootstrap from rayon workers: fhe_sbox_gal_mul_pbs.rs:33-41, main.rs:148-152).  Calls on
 *     one context are serialised by an internal lock; tac_wopbs_coalesced additionally merges concurrent callers into
 *     one batched GPU pass.  tac_last_error() reports the last error of the CALLING thread.
 */
#ifndef TFHE_AES_CUDA_H
#define TFHE_AES_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum tac_status {
    TAC_OK = 0,
    TAC_ERR_CUDA = -1,          /* CUDA runtime error, no device, or the extension was built without kernels */
    TAC_ERR_ARG = -2,           /* bad argument / unsupported parameter set */
    TAC_ERR_STATE = -3,         /* keys not uploaded, unknown LUT id, ... */
    TAC_ERR_NOISE = -4          /* squared-noise budget exceeded (reference: MaxNoiseLevel::validate → NoiseTooBig) */
} tac_status;

/* WopbsParameters + max_noise_level_squared — src/tfhe/shortint_woppbs_1bit/parameters.rs:9-13 */
typedef struct tac_params {
    int32_t lwe_dimension;       /* n */
    int32_t glwe_dimension;      /* k */
    int32_t polynomial_size;     /* N */
    int32_t pbs_level, pbs_base_log;
    int32_t ks_level, ks_base_log;
    int32_t cbs_level, cbs_base_log;
    int32_t pfks_level, pfks_base_log;
    int32_t max_noise_level_squared;
    double lwe_noise_std, glwe_noise_std, pfks_noise_std;
} tac_params;

typedef struct tac_ctx tac_ctx;
typedef struct tac_client_key tac_client_key;

/* ------------------------------------------------------------------ parameters, encodings, LUTs (host, pure integer) */
/* params_sqrd_lvl_{1,4,64,256} — parameters.rs:29-61, :77-109, :125-157, :173-205.  id ∈ {1, 4, 64, 256}. */
int tac_params_preset(int id, tac_params* out);
/* encode_bit / decode_bit — src/tfhe/shortint_woppbs_1bit.rs:125-132 */
uint64_t tac_encode_bit(uint64_t bit);
uint64_t tac_decode_bit(uint64_t encoding);
/* generate_multivariate_luts — shortint_woppbs_1bit.rs:366-403.  f_table[val] = f(val) for val < 2^n_in;
 * out has n_out · tac_lut_len(n_in, N) words. */
size_t tac_lut_len(int n_in, int polynomial_size);
int tac_generate_lut(int n_in, int n_out, int polynomial_size, const uint64_t* f_table, uint64_t* out);

/* ------------------------------------------------------------------ client side (host CPU, like the reference's) */
/* FheContext::generate_keys_with_params — shortint_woppbs_1bit.rs:245-268 (secret keys only; evaluation keys below).
 * tac_client_keygen_os seeds a 256-bit ChaCha20 master key from the OS (getrandom), like the reference (engine.rs:164-168):
 * use it for anything but tests.  tac_client_keygen(p, seed) derives the master key from a 64-bit seed — reproducible,
 * therefore NOT secret: tests and benchmarks only.  Every object (one GLWE / LWE ciphertext) draws from its own stream. */
tac_client_key* tac_client_keygen_os(const tac_params* p);                    /* NULL if the OS entropy source fails */
tac_client_key* tac_client_keygen(const tac_params* p, uint64_t seed);
/* A client around existing secret keys (e.g. loaded with tac_keyfile_*; words must be 0/1); encryption randomness of
 * this instance comes from fresh OS entropy, so masks are never reused across instances. */
tac_client_key* tac_client_from_secret_keys(const tac_params* p, const uint64_t* sk_glwe, const uint64_t* sk_lwe);
void tac_client_free(tac_client_key* ck);
/* which: 0 sk_glwe (kN words, 0/1), 1 sk_lwe (n), 2 BSK standard, 3 KSK, 4 PFPKSK.  Lengths in words. */
size_t tac_key_len(const tac_params* p, int which);
/* [U] shortint::gen_keys + WopbsKey::new_wopbs_key_only_for_wopbs — shortint_woppbs_1bit.rs:246-248.  threads <= 0: all cores. */
int tac_client_gen_eval_keys(tac_client_key* ck, int threads);
const uint64_t* tac_client_key_ptr(tac_client_key* ck, int which);
/* ClientKey::encrypt — shortint_woppbs_1bit.rs:200-217.  Ciphertext i uses RNG stream first_index + i. */
int tac_client_encrypt_bits(tac_client_key* ck, const uint8_t* bits, size_t n, uint64_t first_index, uint64_t* out);
/* ClientKey::decrypt — shortint_woppbs_1bit.rs:219-225 */
int tac_client_decrypt_bits(tac_client_key* ck, const uint64_t* cts, size_t n, uint8_t* bits);
int tac_client_decrypt_phases(tac_client_key* ck, const uint64_t* cts, size_t n, uint64_t* phases);

/* ------------------------------------------------------------------ wire format (csrc/wire.cpp documents the layout) */
/* Flat little-endian dump of the raw `u64` containers the reference obtains from tfhe-rs with into_raw_parts /
 * as_ref() (shortint_woppbs_1bit.rs:245-268): a file written by a tfhe-rs process (INTEGRATION.md has the Rust writer)
 * loads here and vice versa.  Any key pointer may be NULL (section omitted / not read); lengths are tac_key_len(). */
int tac_keys_save(const char* path, const tac_params* p, const uint64_t* sk_glwe, const uint64_t* sk_lwe, const uint64_t* bsk_std,
                  const uint64_t* ksk, const uint64_t* pfpksk);
int tac_keys_load_params(const char* path, tac_params* p, uint32_t* present_mask /* bit i: section id i present */);
int tac_keys_load(const char* path, const tac_params* p, uint64_t* sk_glwe, uint64_t* sk_lwe, uint64_t* bsk_std, uint64_t* ksk, uint64_t* pfpksk);
/* LweCiphertextListOwned<u64>: [count][lwe_size] words.  Load with words == NULL queries the sizes. */
int tac_lwe_list_save(const char* path, uint64_t lwe_size, uint64_t count, const uint64_t* words);
int tac_lwe_list_load(const char* path, uint64_t* lwe_size, uint64_t* count, uint64_t* words, size_t capacity_words);

/* ------------------------------------------------------------------ server context (one per GPU) */
tac_ctx* tac_ctx_create(const tac_params* p, int device);   /* NULL if there is no usable CUDA device */
void tac_ctx_destroy(tac_ctx* ctx);
const char* tac_last_error(tac_ctx* ctx);                   /* ctx may be NULL: error of the last failed create */
int tac_ctx_set_stream(tac_ctx* ctx, void* cuda_stream);    /* cudaStream_t; default: a private non-blocking stream */
int tac_ctx_sync(tac_ctx* ctx);
int tac_ctx_sm_count(tac_ctx* ctx);
/* Evaluation keys (FheContext's server_key + wopbs_key — shortint_woppbs_1bit.rs:166-172).  The BSK is taken in the
 * STANDARD domain and converted on the device. */
int tac_ctx_upload_keys(tac_ctx* ctx, const uint64_t* bsk_std, const uint64_t* ksk, const uint64_t* pfpksk);
int tac_ctx_load_keys(tac_ctx* ctx, const char* key_file);    /* evaluation keys from a tac_keys_save / tfhe-rs-written file */
/* Multi-GPU replication: non-root ranks allocate, every rank exposes its device buffers (which: 0 Fourier BSK, 1 KSK,
 * 2 PFPKSK) to the caller's collective (torch.distributed / ncclBroadcast), then marks them valid. */
int tac_ctx_alloc_keys(tac_ctx* ctx);
int tac_ctx_key_buffer(tac_ctx* ctx, int which, void** dev_ptr, size_t* bytes);
int tac_ctx_keys_ready(tac_ctx* ctx);
/* FheContext::generate_lookup_table result handed to the device — shortint_woppbs_1bit.rs:274-289.  Returns id >= 0. */
int tac_lut_register(tac_ctx* ctx, int n_in, int n_out, const uint64_t* table, size_t len);

/* ------------------------------------------------------------------ the operator */
/* FheContext::circuit_bootstrap — shortint_woppbs_1bit.rs:292-336 — batched: `batch` independent calls with the same LUT.
 * in: [batch][n_in][kN+1], out: [batch][n_out][kN+1].  (extract_dual_bit_from_bit :339-363 = LWE keyswitch;
 * circuit_bootstrapping_vertical_packing :326-328 = PBS + PFKS + GGSW FFT + vertical packing.) */
int tac_wopbs_batch(tac_ctx* ctx, int lut_id, int batch, const uint64_t* in_host, uint64_t* out_host);
int tac_wopbs_batch_dev(tac_ctx* ctx, int lut_id, int batch, const uint64_t* in_dev, uint64_t* out_dev);
/* The same operator for callers that arrive one circuit_bootstrap at a time from many threads — the shape of the
 * reference's rayon fan-out (16 bytes × blocks, fhe_sbox_gal_mul_pbs.rs:33-41): blocks until this request is done;
 * requests that arrive within `window_us` of each other (and while a pass is running) are merged into one batched pass
 * per LUT.  Defaults: window 200 µs, at most 4096 requests per pass. */
int tac_wopbs_coalesced(tac_ctx* ctx, int lut_id, int batch, const uint64_t* in_host, uint64_t* out_host);
int tac_ctx_set_coalescing(tac_ctx* ctx, int window_us, int max_batch);
int tac_ctx_coalescing_stats(tac_ctx* ctx, uint64_t* requests, uint64_t* passes);   /* since creation */
/* BitXorAssign for BitCt — shortint_woppbs_1bit.rs:134-142 (lwe_ciphertext_add_assign); noise bookkeeping stays with the caller */
int tac_lwe_add_batch(tac_ctx* ctx, uint64_t* a_host, const uint64_t* b_host, size_t n_cts);
int tac_lwe_add_batch_dev(tac_ctx* ctx, uint64_t* a_dev, const uint64_t* b_dev, size_t n_cts);

/* ------------------------------------------------------------------ fused AES paths (state stays on the device) */
/* Aes128Encrypt::key_schedule → fhe_sbox_gal_mul_pbs::key_schedule — src/aes_128/fhe/fhe_sbox_gal_mul_pbs.rs:134-164 */
int tac_aes_key_schedule(tac_ctx* ctx, const uint64_t* key_bits_host, uint64_t* key_sched_host);
/* make an expanded key resident on the device (the reference passes &[Word;44] to every encrypt_block call) */
int tac_aes_set_key_schedule(tac_ctx* ctx, const uint64_t* key_sched_host);
int tac_aes_key_schedule_buffer(tac_ctx* ctx, void** dev_ptr, size_t* bytes);   /* for replication to other GPUs */
/* Aes128Encrypt::encrypt_block_for_rounds → fhe_sbox_gal_mul_pbs::encrypt_block_for_rounds — :84-132, over n_blocks
 * independent blocks (main.rs:141-159 runs them with rayon).  in_noise_sq: squared noise level of the input bits
 * (1 for fresh).  Returns TAC_ERR_NOISE where the reference would panic with NoiseTooBig. */
int tac_aes_encrypt_blocks(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_host, uint64_t* out_host);
int tac_aes_encrypt_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_dev, uint64_t* out_dev);
/* Aes128Encrypt::encrypt_block_for_rounds over PUBLIC 16-byte blocks (e.g. AES-CTR counter blocks iv ‖ BE64(ctr),
 * main.rs:108-115) under the device key schedule: state0 = k0 ⊕ trivial(block), no input ciphertexts.  Circuit bootstraps
 * whose inputs are equal across blocks run once: byte j of two blocks shares the round-r S-box when the blocks agree on the
 * input bytes that byte depends on (D(1, j) = {j}, then ShiftRows + MixColumns spread it: a diagonal in round 2, all 16
 * bytes from round 3 on).  Same round structure as tac_aes_encrypt_blocks, including rk10 in the final round.
 *   blocks_host: [n_blocks][16] bytes.  xor_host: NULL, or [n_blocks][16] public bytes XORed into the output — AES-CTR
 *   transciphering: pass the AES-CTR ciphertext and the output encrypts the plaintext.  Both are HOST memory in both
 *   variants.  out: [n_blocks][16][8][kN+1].
 * Output bits carry squared noise level 8 + 1 = 9, as on the encrypted-block path; identical public blocks give
 * word-identical outputs, and the output equals tac_aes_encrypt_blocks on trivial encryptions of the same blocks. */
int tac_aes_encrypt_public_blocks(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_host);
int tac_aes_encrypt_public_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_dev);
/* circuit-bootstrapped S-box boxes per round that tac_aes_encrypt_public_blocks runs for these blocks: boxes[r-1],
 * r = 1..rounds (16·n_blocks each without sharing).  Host only, needs no context or GPU. */
int tac_aes_public_plan(int n_blocks, int rounds, const uint8_t* blocks_host /*[n][16]*/, int64_t* boxes);

/* ------------------------------------------------------------------ AES decryption (no counterpart in the reference) */
/* Inverse key schedule dk of the equivalent inverse cipher (FIPS-197 §5.3.5), derived on the device from the resident
 * encryption schedule w: dk[0..3] = w[0..3], dk[40..43] = w[40..43], dk[4rd..4rd+3] = InvMixColumns(w[4rd..4rd+3]) for
 * rd = 1..9.  Layout as the key schedule, [44 words][4][8][kN+1]; out_host may be NULL.  Runs 144 circuit bootstraps
 * 8 → 32 and 1152 of 1 bit; its bits carry squared noise level 1.  TAC_ERR_NOISE below max_noise_level_squared 32.
 * dk stays valid until the encryption schedule changes: tac_aes_set_key_schedule (and so tac_aes_key_schedule and
 * tac_aes_key_schedule_buffer) marks it stale, and decryption then fails with TAC_ERR_STATE.  No call derives it
 * implicitly. */
int tac_aes_inv_key_schedule(tac_ctx* ctx, uint64_t* inv_key_sched_host);
/* make a given dk resident (e.g. client-encrypted from a clear InvMixColumns schedule); decryption reads every round key,
 * dk[0..3] and dk[40..43] included, from dk only */
int tac_aes_set_inv_key_schedule(tac_ctx* ctx, const uint64_t* inv_key_sched_host);
/* AES decryption of n_blocks blocks with the equivalent inverse cipher: the exact inverse of tac_aes_encrypt_blocks for the
 * same `rounds` (which adds w[40..43] in its final round for every `rounds`):
 *   s = in ⊕ dk[40..43];  rd = rounds−1 … 1: s = InvMixColumns(InvShiftRows(InvS(s))) ⊕ dk[rd];  out = InvShiftRows(InvS(s)) ⊕ dk[0..3]
 * InvS·{14, 11, 13, 9} comes from one 8 → 32 circuit bootstrap per byte.  Noise as in encryption (33 in a middle round,
 * output 9); TAC_ERR_STATE without a valid dk. */
int tac_aes_decrypt_blocks(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_host, uint64_t* out_host);
int tac_aes_decrypt_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, int in_noise_sq, const uint64_t* in_dev, uint64_t* out_dev);
/* decryption of PUBLIC 16-byte ciphertext blocks: state0 = dk[40..43] ⊕ trivial(block).  AES-ECB / AES-CBC transciphering:
 * xor_host NULL (ECB) or the previous ciphertext blocks C_{i-1}, C_{-1} = IV (CBC), and the output encrypts the plaintext.
 * Bootstraps equal across blocks run once, as in tac_aes_encrypt_public_blocks, along the inverse dependence rule
 * D(r+1, (row, c)) = ∪_{r'} D(r, 4·((c − r') mod 4) + r').  Blocks and XOR bytes are HOST memory in both variants; the
 * output equals tac_aes_decrypt_blocks on trivial encryptions of the same blocks. */
int tac_aes_decrypt_public_blocks(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_host);
int tac_aes_decrypt_public_blocks_dev(tac_ctx* ctx, int n_blocks, int rounds, const uint8_t* blocks_host, const uint8_t* xor_host, uint64_t* out_dev);
/* boxes per round that tac_aes_decrypt_public_blocks runs for these blocks (as tac_aes_public_plan).  Host only. */
int tac_aes_public_plan_inv(int n_blocks, int rounds, const uint8_t* blocks_host /*[n][16]*/, int64_t* boxes);

/* ------------------------------------------------------------------ single stages (parity tests, profiling) */
/* [U] keyswitch_lwe_ciphertext: [n_cts][kN+1] → [n_cts][n+1] */
int tac_stage_keyswitch(tac_ctx* ctx, int n_cts, const uint64_t* in_host, uint64_t* out_host);
/* [U] WopbsKey::extract_bits(DeltaLog(delta_log), ct, ExtractedBitsCount(n_bits)) — the general bit-extraction chain
 * (keyswitch → bootstrap of the sign bit → subtract, least significant bit first): [n_cts][kN+1] → [n_cts][n_bits][n+1] under
 * the small key, most significant extracted bit first, each carrying its bit at 2^63.  extract_dual_bit_from_bit
 * (shortint_woppbs_1bit.rs:339-363) is the (63, 1) case = tac_stage_keyswitch; the 8-bit model uses (56, 8)
 * (shortint_woppbs_8bit.rs:271-275). */
int tac_extract_bits(tac_ctx* ctx, int delta_log, int n_bits, int n_cts, const uint64_t* in_host, uint64_t* out_host);
/* [U] homomorphic_shift_boolean: [n_cts][n+1] → [n_cts][kN+1] */
int tac_stage_pbs(tac_ctx* ctx, int n_cts, const uint64_t* in_host, uint64_t* out_host);
/* [U] private_functional_keyswitch ×(k+1): [n_cts][kN+1] → [n_cts][k+1][(k+1)N] */
int tac_stage_pfks(tac_ctx* ctx, int n_cts, const uint64_t* in_host, uint64_t* out_host);
/* [U] vertical_packing from standard-domain GGSWs: ggsw [batch][n_in][cbs_level][k+1][(k+1)N] → [batch][n_out][kN+1] */
int tac_stage_vertical_packing(tac_ctx* ctx, int lut_id, int batch, const uint64_t* ggsw_std_host, uint64_t* out_host);
/* one CMux step  acc += GGSW ⊡ (acc·X^rot − acc)  with a standard-domain GGSW of `levels` levels / base 2^base_log;
 * acc: [n_acc][(k+1)N] in/out, rot[n_acc] in [0, 2N).  Exercises the FFT / external-product core alone. */
int tac_stage_cmux_rotate(tac_ctx* ctx, int levels, int base_log, const uint64_t* ggsw_std_host, int n_acc, const int32_t* rot,
                          uint64_t* acc_host);
/* [U] FourierGgswCiphertext::fill_with_forward_fourier on its own: n_polys torus polynomials [n_polys][N] → Fourier slots
 * [n_polys][N/2] (re, im) doubles, values scaled by 2^-64 · 2/N, in the slot order tac_fft_slot_frequencies reports
 * (slot s holds frequency freq[s] of the size-N/2 FFT of the folded, twisted polynomial). */
int tac_stage_poly_fft(tac_ctx* ctx, size_t n_polys, const uint64_t* polys_host, double* out_host);
int tac_fft_slot_frequencies(int polynomial_size, int32_t* freq /* [N/2] */);
/* [U] extract_lwe_sample_from_glwe_ciphertext(.., MonomialDegree(0)): [n_glwe][(k+1)N] → [n_glwe][kN+1] */
int tac_stage_sample_extract(tac_ctx* ctx, size_t n_glwe, const uint64_t* glwe_host, uint64_t* out_host);
/* Per-stage device time.  With profiling on, every pipeline pass records CUDA events on the context's stream (no host
 * synchronisation); tac_ctx_stage_times synchronises, returns the summed milliseconds since the previous call —
 * [0] keyswitch [1] PBS [2] PFKS [3] GGSW FFT [4] vertical packing — and the number of passes, then resets. */
int tac_ctx_set_profiling(tac_ctx* ctx, int on);
int tac_ctx_stage_times(tac_ctx* ctx, float out_ms[5], int* n_passes);
uint64_t tac_ctx_launch_count(tac_ctx* ctx);                 /* kernels launched since creation */
/* FP64 FMA-pipe throughput of this GPU in TFLOP/s (DFMA microbenchmark): the roofline denominator of the PBS kernel */
int tac_bench_fp64_peak(tac_ctx* ctx, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* TFHE_AES_CUDA_H */
