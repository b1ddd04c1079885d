//! Raw bindings, 1:1 with `include/tfhe_aes_cuda.h`.  Every function returns 0 on success and a negative `tac_status`
//! otherwise; `tac_last_error` gives the message of the calling thread.  All entry points may be called concurrently on
//! one context (the library serialises them; `tac_wopbs_coalesced` merges concurrent callers into one GPU pass).
#![allow(non_camel_case_types)]

use std::os::raw::{c_char, c_int, c_void};

pub const TAC_OK: c_int = 0;
pub const TAC_ERR_CUDA: c_int = -1;
pub const TAC_ERR_ARG: c_int = -2;
pub const TAC_ERR_STATE: c_int = -3;
pub const TAC_ERR_NOISE: c_int = -4;

/// `WopbsParameters` + `max_noise_level_squared` (reference `parameters.rs:9-13`)
#[repr(C)]
#[derive(Clone, Copy, Debug, PartialEq)]
pub struct tac_params {
    pub lwe_dimension: i32,
    pub glwe_dimension: i32,
    pub polynomial_size: i32,
    pub pbs_level: i32,
    pub pbs_base_log: i32,
    pub ks_level: i32,
    pub ks_base_log: i32,
    pub cbs_level: i32,
    pub cbs_base_log: i32,
    pub pfks_level: i32,
    pub pfks_base_log: i32,
    pub max_noise_level_squared: i32,
    pub lwe_noise_std: f64,
    pub glwe_noise_std: f64,
    pub pfks_noise_std: f64,
}

#[repr(C)]
pub struct tac_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct tac_client_key {
    _private: [u8; 0],
}

/// One AES-CCM record (NIST SP 800-38C): `data` = C ‖ U, the ciphertext and the received tag of `tag_len` bytes
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct tac_ccm_msg {
    pub nonce: *const u8,
    pub nonce_len: i32,
    pub tag_len: i32,
    pub aad: *const u8,
    pub aad_len: u64,
    pub data: *const u8,
    pub data_len: u64,
}

extern "C" {
    // parameters, encodings, LUTs
    pub fn tac_params_preset(id: c_int, out: *mut tac_params) -> c_int;
    pub fn tac_encode_bit(bit: u64) -> u64;
    pub fn tac_decode_bit(encoding: u64) -> u64;
    pub fn tac_lut_len(n_in: c_int, polynomial_size: c_int) -> usize;
    pub fn tac_generate_lut(n_in: c_int, n_out: c_int, polynomial_size: c_int, f_table: *const u64, out: *mut u64) -> c_int;

    // client side (optional: a tfhe-rs client can be used instead, see patch/src/tfhe/cuda_woppbs_1bit.rs)
    pub fn tac_client_keygen_os(p: *const tac_params) -> *mut tac_client_key;
    pub fn tac_client_keygen(p: *const tac_params, seed: u64) -> *mut tac_client_key;
    pub fn tac_client_from_secret_keys(p: *const tac_params, sk_glwe: *const u64, sk_lwe: *const u64) -> *mut tac_client_key;
    pub fn tac_client_free(ck: *mut tac_client_key);
    pub fn tac_key_len(p: *const tac_params, which: c_int) -> usize;
    pub fn tac_client_gen_eval_keys(ck: *mut tac_client_key, threads: c_int) -> c_int;
    pub fn tac_client_key_ptr(ck: *mut tac_client_key, which: c_int) -> *const u64;
    pub fn tac_client_encrypt_bits(ck: *mut tac_client_key, bits: *const u8, n: usize, first_index: u64, out: *mut u64) -> c_int;
    pub fn tac_client_decrypt_bits(ck: *mut tac_client_key, cts: *const u64, n: usize, bits: *mut u8) -> c_int;
    pub fn tac_client_decrypt_phases(ck: *mut tac_client_key, cts: *const u64, n: usize, phases: *mut u64) -> c_int;

    // wire format
    pub fn tac_keys_save(path: *const c_char, p: *const tac_params, sk_glwe: *const u64, sk_lwe: *const u64, bsk_std: *const u64,
                         ksk: *const u64, pfpksk: *const u64) -> c_int;
    pub fn tac_keys_load_params(path: *const c_char, p: *mut tac_params, present_mask: *mut u32) -> c_int;
    pub fn tac_keys_load(path: *const c_char, p: *const tac_params, sk_glwe: *mut u64, sk_lwe: *mut u64, bsk_std: *mut u64, ksk: *mut u64,
                         pfpksk: *mut u64) -> c_int;
    pub fn tac_lwe_list_save(path: *const c_char, lwe_size: u64, count: u64, words: *const u64) -> c_int;
    pub fn tac_lwe_list_load(path: *const c_char, lwe_size: *mut u64, count: *mut u64, words: *mut u64, capacity_words: usize) -> c_int;

    // server context
    pub fn tac_ctx_create(p: *const tac_params, device: c_int) -> *mut tac_ctx;
    pub fn tac_ctx_destroy(ctx: *mut tac_ctx);
    pub fn tac_last_error(ctx: *mut tac_ctx) -> *const c_char;
    pub fn tac_ctx_set_stream(ctx: *mut tac_ctx, cuda_stream: *mut c_void) -> c_int;
    pub fn tac_ctx_sync(ctx: *mut tac_ctx) -> c_int;
    pub fn tac_ctx_sm_count(ctx: *mut tac_ctx) -> c_int;
    pub fn tac_ctx_upload_keys(ctx: *mut tac_ctx, bsk_std: *const u64, ksk: *const u64, pfpksk: *const u64) -> c_int;
    pub fn tac_ctx_load_keys(ctx: *mut tac_ctx, key_file: *const c_char) -> c_int;
    pub fn tac_ctx_alloc_keys(ctx: *mut tac_ctx) -> c_int;
    pub fn tac_ctx_key_buffer(ctx: *mut tac_ctx, which: c_int, dev_ptr: *mut *mut c_void, bytes: *mut usize) -> c_int;
    pub fn tac_ctx_keys_ready(ctx: *mut tac_ctx) -> c_int;
    pub fn tac_lut_register(ctx: *mut tac_ctx, n_in: c_int, n_out: c_int, table: *const u64, len: usize) -> c_int;

    // the operator
    pub fn tac_wopbs_batch(ctx: *mut tac_ctx, lut_id: c_int, batch: c_int, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_wopbs_batch_dev(ctx: *mut tac_ctx, lut_id: c_int, batch: c_int, in_dev: *const u64, out_dev: *mut u64) -> c_int;
    pub fn tac_wopbs_coalesced(ctx: *mut tac_ctx, lut_id: c_int, batch: c_int, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_ctx_set_coalescing(ctx: *mut tac_ctx, window_us: c_int, max_batch: c_int) -> c_int;
    pub fn tac_ctx_coalescing_stats(ctx: *mut tac_ctx, requests: *mut u64, passes: *mut u64) -> c_int;
    pub fn tac_lwe_add_batch(ctx: *mut tac_ctx, a_host: *mut u64, b_host: *const u64, n_cts: usize) -> c_int;
    pub fn tac_lwe_add_batch_dev(ctx: *mut tac_ctx, a_dev: *mut u64, b_dev: *const u64, n_cts: usize) -> c_int;

    // fused AES paths
    pub fn tac_aes_key_schedule(ctx: *mut tac_ctx, key_bits_host: *const u64, key_sched_host: *mut u64) -> c_int;
    pub fn tac_aes_set_key_schedule(ctx: *mut tac_ctx, key_sched_host: *const u64) -> c_int;
    pub fn tac_aes_key_schedule_buffer(ctx: *mut tac_ctx, dev_ptr: *mut *mut c_void, bytes: *mut usize) -> c_int;
    pub fn tac_aes_encrypt_blocks(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, in_noise_sq: c_int, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_aes_encrypt_blocks_dev(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, in_noise_sq: c_int, in_dev: *const u64, out_dev: *mut u64) -> c_int;
    pub fn tac_aes_encrypt_public_blocks(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, blocks_host: *const u8, xor_host: *const u8, out_host: *mut u64) -> c_int;
    pub fn tac_aes_encrypt_public_blocks_dev(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, blocks_host: *const u8, xor_host: *const u8, out_dev: *mut u64) -> c_int;
    pub fn tac_aes_public_plan(n_blocks: c_int, rounds: c_int, blocks_host: *const u8, boxes: *mut i64) -> c_int;
    pub fn tac_aes_inv_key_schedule(ctx: *mut tac_ctx, inv_key_sched_host: *mut u64) -> c_int;
    pub fn tac_aes_set_inv_key_schedule(ctx: *mut tac_ctx, inv_key_sched_host: *const u64) -> c_int;
    pub fn tac_aes_decrypt_blocks(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, in_noise_sq: c_int, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_aes_decrypt_blocks_dev(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, in_noise_sq: c_int, in_dev: *const u64, out_dev: *mut u64) -> c_int;
    pub fn tac_aes_decrypt_public_blocks(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, blocks_host: *const u8, xor_host: *const u8, out_host: *mut u64) -> c_int;
    pub fn tac_aes_decrypt_public_blocks_dev(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, blocks_host: *const u8, xor_host: *const u8, out_dev: *mut u64) -> c_int;
    pub fn tac_aes_public_plan_inv(n_blocks: c_int, rounds: c_int, blocks_host: *const u8, boxes: *mut i64) -> c_int;
    // AES under many keys (no counterpart in the reference)
    pub fn tac_aes_key_table(ctx: *mut tac_ctx, n_keys: c_int, key_bits_host: *const u64, key_scheds_host: *mut u64) -> c_int;
    pub fn tac_aes_set_key_table(ctx: *mut tac_ctx, n_keys: c_int, key_scheds_host: *const u64) -> c_int;
    pub fn tac_aes_inv_key_table(ctx: *mut tac_ctx, inv_key_scheds_host: *mut u64) -> c_int;
    pub fn tac_aes_set_inv_key_table(ctx: *mut tac_ctx, inv_key_scheds_host: *const u64) -> c_int;
    pub fn tac_aes_encrypt_blocks_keyed(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, in_noise_sq: c_int, key_idx_host: *const i32, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_aes_encrypt_blocks_keyed_dev(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, in_noise_sq: c_int, key_idx_host: *const i32, in_dev: *const u64, out_dev: *mut u64) -> c_int;
    pub fn tac_aes_decrypt_blocks_keyed(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, in_noise_sq: c_int, key_idx_host: *const i32, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_aes_decrypt_blocks_keyed_dev(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, in_noise_sq: c_int, key_idx_host: *const i32, in_dev: *const u64, out_dev: *mut u64) -> c_int;
    pub fn tac_aes_encrypt_public_blocks_keyed(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, key_idx_host: *const i32, blocks_host: *const u8, xor_host: *const u8, out_host: *mut u64) -> c_int;
    pub fn tac_aes_encrypt_public_blocks_keyed_dev(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, key_idx_host: *const i32, blocks_host: *const u8, xor_host: *const u8, out_dev: *mut u64) -> c_int;
    pub fn tac_aes_decrypt_public_blocks_keyed(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, key_idx_host: *const i32, blocks_host: *const u8, xor_host: *const u8, out_host: *mut u64) -> c_int;
    pub fn tac_aes_decrypt_public_blocks_keyed_dev(ctx: *mut tac_ctx, n_blocks: c_int, rounds: c_int, key_idx_host: *const i32, blocks_host: *const u8, xor_host: *const u8, out_dev: *mut u64) -> c_int;
    pub fn tac_aes_public_plan_keyed(n_blocks: c_int, rounds: c_int, decrypt: c_int, key_idx: *const i32, blocks_host: *const u8, boxes: *mut i64) -> c_int;
    // AES-CCM transciphering with the tag checked under FHE (no counterpart in the reference)
    pub fn tac_aes_ccm_transcipher(ctx: *mut tac_ctx, n_msgs: c_int, key_idx: *const i32, msgs: *const tac_ccm_msg, pt_out_host: *mut u64,
                                   valid_out_host: *mut u64) -> c_int;
    pub fn tac_aes_ccm_transcipher_dev(ctx: *mut tac_ctx, n_msgs: c_int, key_idx: *const i32, msgs: *const tac_ccm_msg, pt_out_dev: *mut u64,
                                       valid_out_dev: *mut u64) -> c_int;
    pub fn tac_aes_ccm_format(msg: *const tac_ccm_msg, ctr_blocks: *mut u8, mac_blocks: *mut u8, counts: *mut i64) -> c_int;
    pub fn tac_aes_gcm_hash_key(ctx: *mut tac_ctx, depth: c_int, out_host: *mut u64) -> c_int;
    pub fn tac_aes_gcm_hash_key_table(ctx: *mut tac_ctx, depth: c_int, out_host: *mut u64) -> c_int;
    pub fn tac_aes_gcm_transcipher(ctx: *mut tac_ctx, n_msgs: c_int, key_idx: *const i32, msgs: *const tac_ccm_msg, pt_out_host: *mut u64,
                                   valid_out_host: *mut u64) -> c_int;
    pub fn tac_aes_gcm_transcipher_dev(ctx: *mut tac_ctx, n_msgs: c_int, key_idx: *const i32, msgs: *const tac_ccm_msg, pt_out_dev: *mut u64,
                                       valid_out_dev: *mut u64) -> c_int;
    pub fn tac_aes_gcm_format(msg: *const tac_ccm_msg, ctr_blocks: *mut u8, ghash_blocks: *mut u8, counts: *mut i64) -> c_int;
    pub fn tac_gf128_mul(ctx: *mut tac_ctx, n: c_int, a_host: *const u64, b_host: *const u64, out_host: *mut u64) -> c_int;

    // single stages, profiling
    pub fn tac_stage_keyswitch(ctx: *mut tac_ctx, n_cts: c_int, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_extract_bits(ctx: *mut tac_ctx, delta_log: c_int, n_bits: c_int, n_cts: c_int, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_stage_pbs(ctx: *mut tac_ctx, n_cts: c_int, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_stage_pfks(ctx: *mut tac_ctx, n_cts: c_int, in_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_stage_vertical_packing(ctx: *mut tac_ctx, lut_id: c_int, batch: c_int, ggsw_std_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_stage_cmux_rotate(ctx: *mut tac_ctx, levels: c_int, base_log: c_int, ggsw_std_host: *const u64, n_acc: c_int, rot: *const i32,
                                 acc_host: *mut u64) -> c_int;
    pub fn tac_stage_poly_fft(ctx: *mut tac_ctx, n_polys: usize, polys_host: *const u64, out_host: *mut f64) -> c_int;
    pub fn tac_fft_slot_frequencies(polynomial_size: c_int, freq: *mut i32) -> c_int;
    pub fn tac_stage_sample_extract(ctx: *mut tac_ctx, n_glwe: usize, glwe_host: *const u64, out_host: *mut u64) -> c_int;
    pub fn tac_ctx_set_profiling(ctx: *mut tac_ctx, on: c_int) -> c_int;
    pub fn tac_ctx_stage_times(ctx: *mut tac_ctx, out_ms: *mut f32, n_passes: *mut c_int) -> c_int;
    pub fn tac_ctx_launch_count(ctx: *mut tac_ctx) -> u64;
    pub fn tac_bench_fp64_peak(ctx: *mut tac_ctx, tflops: *mut f64) -> c_int;
}
