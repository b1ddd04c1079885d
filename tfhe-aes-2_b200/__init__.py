"""tfhe-aes-2_b200 — host-side mirror of the reference's `shortint_woppbs_1bit` model on top of the C ABI
(include/tfhe_aes_cuda.h, built from csrc/ into csrc/libtfhe_aes_cuda.so).

Names follow the reference (src/tfhe/shortint_woppbs_1bit.rs): `FheContext`, `ClientKey`, `BitCt`, `encode_bit`,
`decode_bit`, `generate_lookup_table`, `circuit_bootstrap`; the noise bookkeeping (`NoiseLevelWithComponents`, :35-78)
lives here on the host exactly as in the reference, the lattice arithmetic runs on the GPU.  There is no CPU fallback:
importing works without a GPU (so that the client side and the pure-integer helpers are usable), creating an
`FheContext` without the built extension or without a B200 raises.

The directory name is not a Python identifier; import it with
    importlib.import_module("tfhe-aes-2_b200")
"""
import ctypes as C
import itertools
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "csrc", "libtfhe_aes_cuda.so")

TAC_OK, TAC_ERR_CUDA, TAC_ERR_ARG, TAC_ERR_STATE, TAC_ERR_NOISE = 0, -1, -2, -3, -4


class NoiseTooBig(RuntimeError):
    """reference: MaxNoiseLevel::validate(..).unwrap() panics with NoiseTooBig (shortint_woppbs_1bit.rs:74-76)"""


class Params(C.Structure):
    """WopbsParameters + max_noise_level_squared (reference parameters.rs:9-13); layout of `tac_params`."""
    _fields_ = [
        ("lwe_dimension", C.c_int32), ("glwe_dimension", C.c_int32), ("polynomial_size", C.c_int32),
        ("pbs_level", C.c_int32), ("pbs_base_log", C.c_int32),
        ("ks_level", C.c_int32), ("ks_base_log", C.c_int32),
        ("cbs_level", C.c_int32), ("cbs_base_log", C.c_int32),
        ("pfks_level", C.c_int32), ("pfks_base_log", C.c_int32),
        ("max_noise_level_squared", C.c_int32),
        ("lwe_noise_std", C.c_double), ("glwe_noise_std", C.c_double), ("pfks_noise_std", C.c_double),
    ]

    @property
    def big_lwe_dimension(self):
        return self.glwe_dimension * self.polynomial_size

    @property
    def big_lwe_size(self):
        return self.big_lwe_dimension + 1


_lib = None
_u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")

# every symbol include/tfhe_aes_cuda.h declares: (restype, argtypes)
_SIGNATURES = {
    "tac_params_preset": (C.c_int, [C.c_int, C.POINTER(Params)]),
    "tac_encode_bit": (C.c_uint64, [C.c_uint64]),
    "tac_decode_bit": (C.c_uint64, [C.c_uint64]),
    "tac_lut_len": (C.c_size_t, [C.c_int, C.c_int]),
    "tac_generate_lut": (C.c_int, [C.c_int, C.c_int, C.c_int, _u64p, _u64p]),
    "tac_client_keygen": (C.c_void_p, [C.POINTER(Params), C.c_uint64]),
    "tac_client_keygen_os": (C.c_void_p, [C.POINTER(Params)]),
    "tac_client_from_secret_keys": (C.c_void_p, [C.POINTER(Params), _u64p, _u64p]),
    "tac_client_free": (None, [C.c_void_p]),
    "tac_key_len": (C.c_size_t, [C.POINTER(Params), C.c_int]),
    "tac_client_gen_eval_keys": (C.c_int, [C.c_void_p, C.c_int]),
    "tac_client_key_ptr": (C.POINTER(C.c_uint64), [C.c_void_p, C.c_int]),
    "tac_client_encrypt_bits": (C.c_int, [C.c_void_p, _u8p, C.c_size_t, C.c_uint64, _u64p]),
    "tac_client_decrypt_bits": (C.c_int, [C.c_void_p, _u64p, C.c_size_t, _u8p]),
    "tac_client_decrypt_phases": (C.c_int, [C.c_void_p, _u64p, C.c_size_t, _u64p]),
    "tac_keys_save": (C.c_int, [C.c_char_p, C.POINTER(Params), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_keys_load_params": (C.c_int, [C.c_char_p, C.POINTER(Params), C.POINTER(C.c_uint32)]),
    "tac_keys_load": (C.c_int, [C.c_char_p, C.POINTER(Params), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_lwe_list_save": (C.c_int, [C.c_char_p, C.c_uint64, C.c_uint64, C.c_void_p]),
    "tac_lwe_list_load": (C.c_int, [C.c_char_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_void_p, C.c_size_t]),
    "tac_ctx_load_keys": (C.c_int, [C.c_void_p, C.c_char_p]),
    "tac_ctx_create": (C.c_void_p, [C.POINTER(Params), C.c_int]),
    "tac_ctx_destroy": (None, [C.c_void_p]),
    "tac_last_error": (C.c_char_p, [C.c_void_p]),
    "tac_ctx_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tac_ctx_sync": (C.c_int, [C.c_void_p]),
    "tac_ctx_sm_count": (C.c_int, [C.c_void_p]),
    "tac_ctx_upload_keys": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_ctx_alloc_keys": (C.c_int, [C.c_void_p]),
    "tac_ctx_key_buffer": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "tac_ctx_keys_ready": (C.c_int, [C.c_void_p]),
    "tac_lut_register": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _u64p, C.c_size_t]),
    "tac_wopbs_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_wopbs_batch_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_wopbs_coalesced": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_ctx_set_coalescing": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "tac_ctx_coalescing_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "tac_lwe_add_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tac_lwe_add_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tac_aes_key_schedule": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_set_key_schedule": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tac_aes_key_schedule_buffer": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "tac_aes_encrypt_blocks": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_aes_encrypt_blocks_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_aes_encrypt_public_blocks": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_encrypt_public_blocks_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_public_plan": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_aes_inv_key_schedule": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tac_aes_set_inv_key_schedule": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tac_aes_decrypt_blocks": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_aes_decrypt_blocks_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_aes_decrypt_public_blocks": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_decrypt_public_blocks_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_public_plan_inv": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_aes_key_table": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "tac_aes_set_key_table": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "tac_aes_inv_key_table": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tac_aes_set_inv_key_table": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tac_aes_encrypt_blocks_keyed": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_encrypt_blocks_keyed_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_decrypt_blocks_keyed": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_decrypt_blocks_keyed_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_encrypt_public_blocks_keyed": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_encrypt_public_blocks_keyed_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_decrypt_public_blocks_keyed": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_decrypt_public_blocks_keyed_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_public_plan_keyed": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_ccm_transcipher": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_ccm_transcipher_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_ccm_format": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_gcm_hash_key": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "tac_aes_gcm_hash_key_table": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "tac_aes_gcm_transcipher": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_gcm_transcipher_dev": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_aes_gcm_format": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tac_gf128_mul": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p, _u64p]),
    "tac_stage_keyswitch": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p]),
    "tac_extract_bits": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, _u64p, _u64p]),
    "tac_stage_pbs": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p]),
    "tac_stage_pfks": (C.c_int, [C.c_void_p, C.c_int, _u64p, _u64p]),
    "tac_stage_vertical_packing": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _u64p, _u64p]),
    "tac_stage_cmux_rotate": (C.c_int, [C.c_void_p, C.c_int, C.c_int, _u64p, C.c_int, _i32p, _u64p]),
    "tac_stage_poly_fft": (C.c_int, [C.c_void_p, C.c_size_t, _u64p, np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")]),
    "tac_fft_slot_frequencies": (C.c_int, [C.c_int, _i32p]),
    "tac_stage_sample_extract": (C.c_int, [C.c_void_p, C.c_size_t, _u64p, _u64p]),
    "tac_ctx_set_profiling": (C.c_int, [C.c_void_p, C.c_int]),
    "tac_ctx_stage_times": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "tac_bench_fp64_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "tac_ctx_launch_count": (C.c_uint64, [C.c_void_p]),
}


def library_path():
    return _SO


def load_library():
    """Load the sm_100a extension.  Fails loudly when it has not been built (`__graft_entry__.build()`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise RuntimeError(f"CUDA extension not built: {_SO} is missing (run `python -c 'import __graft_entry__ as g; g.build()'`); "
                           "there is no CPU fallback")
    L = C.CDLL(_SO)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(L, name)          # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def params_preset(pid):
    """params_sqrd_lvl_{1,4,64,256} (reference parameters.rs:29-205)."""
    p = Params()
    if load_library().tac_params_preset(pid, C.byref(p)) != 0:
        raise ValueError(f"unknown parameter preset {pid}")
    return p


def encode_bit(bit):
    """reference shortint_woppbs_1bit.rs:125-128"""
    assert bit < 2, f"cleartext out of bounds: {bit}"
    return int(load_library().tac_encode_bit(bit))


def decode_bit(encoding):
    """reference shortint_woppbs_1bit.rs:130-132"""
    return int(load_library().tac_decode_bit(encoding))


def u8_to_bits(byte):
    """MSB first (reference src/util.rs:33-35)"""
    return [0 if 0 == (byte & (0x80 >> i)) else 1 for i in range(8)]


def bits_to_u8(bits):
    """reference src/util.rs:37-42"""
    return sum(int(b) << (7 - i) for i, b in enumerate(bits))


def u16_to_bits(word):
    return [0 if 0 == (word & (0x8000 >> i)) else 1 for i in range(16)]


def generate_multivariate_luts(input_bits, output_bits, polynomial_size, f):
    """reference shortint_woppbs_1bit.rs:366-403; returns a [output_bits][N << tree_bits] uint64 array."""
    assert 0 < input_bits <= 16
    assert 0 < output_bits <= 64
    L = load_library()
    table = np.array([int(f(v)) & 0xFFFFFFFFFFFFFFFF for v in range(1 << input_bits)], dtype=np.uint64)
    out = np.empty((output_bits, L.tac_lut_len(input_bits, polynomial_size)), dtype=np.uint64)
    rc = L.tac_generate_lut(input_bits, output_bits, polynomial_size, table, out)
    if rc != 0:
        raise ValueError("generate_lut: bad arguments")
    return out


def save_lwe_list(path, cts):
    """LweCiphertextListOwned<u64> as a wire file: cts is [count][lwe_size] (any leading shape is flattened)"""
    a = np.ascontiguousarray(cts, dtype=np.uint64)
    a = a.reshape(-1, a.shape[-1])
    if load_library().tac_lwe_list_save(os.fsencode(path), a.shape[1], a.shape[0], a.ctypes.data) != 0:
        raise OSError(f"cannot write {path}")


def load_lwe_list(path):
    L = load_library()
    size, count = C.c_uint64(), C.c_uint64()
    if L.tac_lwe_list_load(os.fsencode(path), C.byref(size), C.byref(count), None, 0) != 0:
        raise OSError(f"{path}: not an LWE list file")
    out = np.empty((count.value, size.value), dtype=np.uint64)
    if L.tac_lwe_list_load(os.fsencode(path), None, None, out.ctypes.data, out.size) != 0:
        raise OSError(f"{path}: truncated or corrupted")
    return out


def key_file_info(path):
    """(Params, set of section ids) of a key file"""
    p, mask = Params(), C.c_uint32()
    if load_library().tac_keys_load_params(os.fsencode(path), C.byref(p), C.byref(mask)) != 0:
        raise OSError(f"{path}: not a key file")
    return p, {i for i in range(32) if mask.value >> i & 1}


def _public_blocks(blocks):
    """[n][16] uint8 from an array, a list of 16-byte strings or one byte string of 16·n bytes"""
    if isinstance(blocks, (bytes, bytearray, memoryview)):
        blocks = np.frombuffer(bytes(blocks), dtype=np.uint8)
    elif not isinstance(blocks, np.ndarray):
        blocks = np.frombuffer(b"".join(bytes(b) for b in blocks), dtype=np.uint8)
    b = np.ascontiguousarray(blocks, dtype=np.uint8)
    if b.size % 16:
        raise ValueError("public blocks must be whole 16-byte blocks")
    return b.reshape(-1, 16)


def ctr_blocks(iv, first_ctr, n):
    """AES-CTR counter blocks iv ‖ BE64(first_ctr + i), i < n (reference main.rs:108-115): [n][16] uint8"""
    iv = bytes(iv)
    if len(iv) != 8:
        raise ValueError("iv must be 8 bytes")
    if n < 0 or first_ctr < 0 or first_ctr + n > 1 << 64:
        raise ValueError("counter range must lie in [0, 2^64)")
    return _public_blocks(b"".join(iv + (first_ctr + i).to_bytes(8, "big") for i in range(n)))


def _key_index(key_index, n_blocks, n_keys=None):
    """int32 [n_blocks] from a sequence of key indices; with n_keys, every index must lie in [0, n_keys)"""
    if key_index is None:
        raise ValueError("a key index per block is required")
    k = np.asarray(key_index)
    if k.size and not np.issubdtype(k.dtype, np.integer):
        raise ValueError("key indices must be integers")
    k = np.ascontiguousarray(k, dtype=np.int64).ravel()
    if k.size != n_blocks:
        raise ValueError(f"{k.size} key indices for {n_blocks} blocks")
    if k.size and (k.min() < 0 or (n_keys is not None and k.max() >= n_keys)):
        raise ValueError(f"key index outside [0, {n_keys})")
    return k.astype(np.int32)


def aes_public_plan(blocks, rounds=10, decrypt=False, key_index=None):
    """circuit bootstraps per round that FheContext.aes_encrypt_public_blocks (decrypt=True: aes_decrypt_public_blocks) runs
    for these public blocks (rounds 1..rounds); 16 per block and round without sharing.  key_index: the keyed paths' plan
    (aes_encrypt_public_blocks_keyed / aes_decrypt_public_blocks_keyed), where only blocks of the same key share.  Host only."""
    b = _public_blocks(blocks)
    out = np.zeros(max(rounds, 0), dtype=np.int64)
    L = load_library()
    if key_index is None:
        plan = L.tac_aes_public_plan_inv if decrypt else L.tac_aes_public_plan
        rc = plan(b.shape[0], rounds, b.ctypes.data, out.ctypes.data)
    else:
        k = np.ascontiguousarray(np.asarray(key_index, dtype=np.int64).ravel(), dtype=np.int32)
        if k.size != b.shape[0]:
            raise ValueError(f"{k.size} key indices for {b.shape[0]} blocks")
        rc = L.tac_aes_public_plan_keyed(b.shape[0], rounds, int(decrypt), k.ctypes.data, b.ctypes.data, out.ctypes.data)
    if rc != 0:
        raise ValueError(f"aes_public_plan: rounds must be in 1..10 and key indices non-negative (error {rc})")
    return [int(v) for v in out]


CCM_TAG_LENGTHS = (4, 6, 8, 10, 12, 14, 16)


class CcmMsg(C.Structure):
    """one AES-CCM record, layout of `tac_ccm_msg`: data = C ‖ U (ciphertext, then the received tag)"""
    _fields_ = [
        ("nonce", C.c_void_p), ("nonce_len", C.c_int32), ("tag_len", C.c_int32),
        ("aad", C.c_void_p), ("aad_len", C.c_uint64),
        ("data", C.c_void_p), ("data_len", C.c_uint64),
    ]


def _ccm_messages(messages):
    """(CcmMsg array, the byte strings it points into, payload length of every message) from [(nonce, data, tag_len, aad)];
    ValueError for every argument the C entry points reject with TAC_ERR_ARG"""
    msgs = (CcmMsg * max(1, len(messages)))()
    keep, sizes = [], []
    for i, (nonce, data, tag_len, aad) in enumerate(messages):
        nonce, data, aad = bytes(nonce), bytes(data), bytes(aad)
        if not 7 <= len(nonce) <= 13:
            raise ValueError(f"AES-CCM message {i}: the nonce must be 7..13 bytes, not {len(nonce)}")
        if not isinstance(tag_len, (int, np.integer)) or int(tag_len) not in CCM_TAG_LENGTHS:
            raise ValueError(f"AES-CCM message {i}: tag length {tag_len!r} not in {CCM_TAG_LENGTHS}")
        tag_len = int(tag_len)
        if len(data) < tag_len:
            raise ValueError(f"AES-CCM message {i}: {len(data)} data bytes cannot hold a {tag_len}-byte tag")
        q, p = 15 - len(nonce), len(data) - tag_len
        if q < 8 and p >> (8 * q):
            raise ValueError(f"AES-CCM message {i}: a payload of {p} bytes does not fit the {q}-byte length field of a {len(nonce)}-byte nonce")
        keep += [nonce, data, aad]
        ptr = lambda b: C.cast(C.c_char_p(b), C.c_void_p).value
        msgs[i] = CcmMsg(ptr(nonce), len(nonce), tag_len, ptr(aad), len(aad), ptr(data), len(data))
        sizes.append(p)
    return msgs, keep, sizes


def aes_ccm_format(nonce, data, tag_len=16, aad=b""):
    """the public blocks of one AES-CCM record (NIST SP 800-38C): (counter blocks A_0..A_m [m+1][16], CBC-MAC blocks
    [B_0, AAD blocks, m zero blocks that stand for the plaintext] [n][16]) as uint8 arrays; data = C ‖ U.  Host only."""
    msgs, keep, _ = _ccm_messages([(nonce, data, tag_len, aad)])
    L = load_library()
    counts = np.zeros(2, dtype=np.int64)
    if L.tac_aes_ccm_format(C.addressof(msgs[0]), None, None, counts.ctypes.data) != 0:
        raise ValueError("aes_ccm_format: bad arguments")
    ctr = np.zeros((int(counts[0]), 16), dtype=np.uint8)
    mac = np.zeros((int(counts[1]), 16), dtype=np.uint8)
    if L.tac_aes_ccm_format(C.addressof(msgs[0]), ctr.ctypes.data, mac.ctypes.data, counts.ctypes.data) != 0:
        raise ValueError("aes_ccm_format: bad arguments")
    return ctr, mac


GCM_TAG_LENGTHS = (4, 8, 12, 13, 14, 15, 16)


def _gcm_messages(messages):
    """(CcmMsg array, the byte strings it points into, payload length of every record) from [(iv, data, tag_len, aad)];
    ValueError for every argument the C entry points reject with TAC_ERR_ARG"""
    msgs = (CcmMsg * max(1, len(messages)))()
    keep, sizes = [], []
    for i, (iv, data, tag_len, aad) in enumerate(messages):
        iv, data, aad = bytes(iv), bytes(data), bytes(aad)
        if len(iv) != 12:
            raise ValueError(f"AES-GCM record {i}: the IV must be 12 bytes, not {len(iv)}")
        if not isinstance(tag_len, (int, np.integer)) or int(tag_len) not in GCM_TAG_LENGTHS:
            raise ValueError(f"AES-GCM record {i}: tag length {tag_len!r} not in {GCM_TAG_LENGTHS}")
        tag_len = int(tag_len)
        if len(data) < tag_len:
            raise ValueError(f"AES-GCM record {i}: {len(data)} data bytes cannot hold a {tag_len}-byte tag")
        p = len(data) - tag_len
        if p > (1 << 36) - 32 or len(aad) >= 1 << 61:
            raise ValueError(f"AES-GCM record {i}: a payload above 2^36 - 32 bytes or AAD of 2^61 bytes or more")
        keep += [iv, data, aad]
        ptr = lambda b: C.cast(C.c_char_p(b), C.c_void_p).value
        msgs[i] = CcmMsg(ptr(iv), len(iv), tag_len, ptr(aad), len(aad), ptr(data), len(data))
        sizes.append(p)
    return msgs, keep, sizes


def aes_gcm_format(iv, data, tag_len=16, aad=b""):
    """the public blocks of one AES-GCM record (NIST SP 800-38D, 96-bit IV): (counter blocks J0, inc32(J0), …
    [m+1][16], GHASH blocks X_1..X_M [M][16]: AAD and C zero-padded, then the bit lengths) as uint8 arrays; data = C ‖ T.
    Host only."""
    msgs, keep, _ = _gcm_messages([(iv, data, tag_len, aad)])
    L = load_library()
    counts = np.zeros(2, dtype=np.int64)
    if L.tac_aes_gcm_format(C.addressof(msgs[0]), None, None, counts.ctypes.data) != 0:
        raise ValueError("aes_gcm_format: bad arguments")
    ctr = np.zeros((int(counts[0]), 16), dtype=np.uint8)
    ghash = np.zeros((int(counts[1]), 16), dtype=np.uint8)
    if L.tac_aes_gcm_format(C.addressof(msgs[0]), ctr.ctypes.data, ghash.ctypes.data, counts.ctypes.data) != 0:
        raise ValueError("aes_gcm_format: bad arguments")
    return ctr, ghash


def _gcm_depth(depth):
    if not isinstance(depth, (int, np.integer)) or not 1 <= int(depth) <= 1024 or int(depth) & (int(depth) - 1):
        raise ValueError(f"GHASH key depth must be a power of two in [1, 1024], not {depth!r}")
    return int(depth)


class LookupTable:
    """WopbsLUTBase plus its shape; registered on the device on first use."""

    def __init__(self, table, input_bits, output_bits):
        self.table = np.ascontiguousarray(table, dtype=np.uint64)
        self.input_bits, self.output_bits = input_bits, output_bits
        self._ids = {}

    def device_id(self, ctx):
        key = ctx._token          # unique per FheContext for the life of the process (id() can be reused after garbage collection)
        if key not in self._ids:
            rc = ctx.L.tac_lut_register(ctx.h, self.input_bits, self.output_bits, self.table.reshape(-1), self.table.size)
            if rc < 0:
                raise RuntimeError(ctx.last_error())
            self._ids[key] = rc
        return self._ids[key]


class _OwnedArray(np.ndarray):
    """view of C-owned key memory that keeps its owner (the ClientKey) alive"""
    _owner = None


class ClientKey:
    """reference ClientKey (shortint_woppbs_1bit.rs:189-226): holds the secret keys, encrypts/decrypts bits on the CPU.

    seed=None (default): all key material and encryption randomness derive from 256 bits of OS entropy, like the
    reference (engine.rs:164-168).  An integer seed gives reproducible — hence publicly computable — keys: tests and
    benchmarks only.  `secret_keys=(sk_glwe, sk_lwe)` wraps existing keys (see save_keys / load_keys)."""

    def __init__(self, params, seed=None, secret_keys=None):
        self.L = load_library()
        self.params = params if isinstance(params, Params) else params_preset(params)
        self.seed = seed
        if secret_keys is not None:
            g, l = (np.ascontiguousarray(a, dtype=np.uint64) for a in secret_keys)
            assert g.size == self.params.big_lwe_dimension and l.size == self.params.lwe_dimension
            self.h = self.L.tac_client_from_secret_keys(C.byref(self.params), g, l)
        elif seed is None:
            self.h = self.L.tac_client_keygen_os(C.byref(self.params))
        else:
            self.h = self.L.tac_client_keygen(C.byref(self.params), seed)
        if not self.h:
            raise RuntimeError("client key creation failed (OS entropy source unavailable, or secret key words not 0/1)")
        self._next_index = itertools.count()
        self._lock = threading.Lock()
        self._enc_counter = 0
        self.context = NoiseContext(self.params)

    def __del__(self):
        try:
            if self.h:
                self.L.tac_client_free(self.h)
                self.h = None
        except Exception:
            pass

    def _key(self, which):
        ptr = self.L.tac_client_key_ptr(self.h, which)
        if not ptr:
            raise RuntimeError("evaluation keys not generated yet (gen_eval_keys)")
        arr = np.ctypeslib.as_array(ptr, shape=(self.L.tac_key_len(C.byref(self.params), which),)).view(_OwnedArray)
        arr._owner = self          # the memory belongs to the C object tac_client_free releases in __del__
        return arr

    def gen_eval_keys(self, threads=0):
        rc = self.L.tac_client_gen_eval_keys(self.h, threads)
        assert rc == 0
        return self

    sk_glwe = property(lambda self: self._key(0))
    sk_lwe = property(lambda self: self._key(1))
    bsk = property(lambda self: self._key(2))
    ksk = property(lambda self: self._key(3))
    pfpksk = property(lambda self: self._key(4))

    # -- wire format (csrc/wire.cpp): the raw tfhe-rs containers, so keys can come from / go to a reference build
    def save_keys(self, path, secret=False, evaluation=True):
        ptr = lambda which, on: self._key(which).ctypes.data if on else None
        rc = self.L.tac_keys_save(os.fsencode(path), C.byref(self.params), ptr(0, secret), ptr(1, secret), ptr(2, evaluation), ptr(3, evaluation),
                                  ptr(4, evaluation))
        if rc != 0:
            raise OSError(f"cannot write {path}")

    @classmethod
    def load_secret_keys(cls, path):
        """a client around the secret keys of a key file (sections 1 and 2); encryption randomness is fresh OS entropy"""
        p, present = key_file_info(path)
        if not {1, 2} <= present:
            raise OSError(f"{path} holds no secret keys")
        L = load_library()
        g, l = np.empty(L.tac_key_len(C.byref(p), 0), dtype=np.uint64), np.empty(L.tac_key_len(C.byref(p), 1), dtype=np.uint64)
        if L.tac_keys_load(os.fsencode(path), C.byref(p), g.ctypes.data, l.ctypes.data, None, None, None) != 0:
            raise OSError(f"{path}: truncated or corrupted")
        return cls(p, secret_keys=(g, l))

    # -- raw array API
    def encrypt_bits(self, bits, first_index=None):
        bits = np.ascontiguousarray(bits, dtype=np.uint8).ravel()
        with self._lock:
            if first_index is None:
                first_index = self._enc_counter
            self._enc_counter = max(self._enc_counter, first_index + bits.size)
        out = np.empty((bits.size, self.params.big_lwe_size), dtype=np.uint64)
        rc = self.L.tac_client_encrypt_bits(self.h, bits, bits.size, first_index, out)
        if rc != 0:
            raise AssertionError("cleartext out of bounds")
        return out

    def encrypt_bytes(self, data, first_index=None):
        bits = [b for v in bytes(data) for b in u8_to_bits(v)]
        return self.encrypt_bits(bits, first_index).reshape(len(data), 8, self.params.big_lwe_size)

    def decrypt_phases(self, cts):
        cts = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, self.params.big_lwe_size)
        out = np.empty(cts.shape[0], dtype=np.uint64)
        self.L.tac_client_decrypt_phases(self.h, cts, cts.shape[0], out)
        return out

    def decrypt_bits(self, cts):
        cts = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, self.params.big_lwe_size)
        out = np.empty(cts.shape[0], dtype=np.uint8)
        self.L.tac_client_decrypt_bits(self.h, cts, cts.shape[0], out)
        return out

    def decrypt_bytes(self, cts):
        bits = self.decrypt_bits(cts).reshape(-1, 8)
        return bytes(bits_to_u8(r) for r in bits)

    # -- ClientKeyT (reference src/tfhe.rs:11-17)
    def encrypt(self, bit):
        assert bit < 2, f"cleartext out of bounds: {bit}"
        return BitCt.fresh(self.encrypt_bits([bit])[0], self.context)

    def decrypt(self, bit_ct):
        return int(self.decrypt_bits(bit_ct.ct)[0])


class NoiseLevelWithComponents:
    """reference shortint_woppbs_1bit.rs:35-78"""
    __slots__ = ("noise_level_squared", "components")

    def __init__(self, noise_level_squared, components):
        self.noise_level_squared = noise_level_squared
        self.components = components

    @classmethod
    def with_noise_level(cls, noise_level_squared, ct_id):
        return cls(noise_level_squared, {ct_id})

    @classmethod
    def trivial(cls):
        return cls(0, set())

    def add_assign(self, rhs, max_noise_level_squared):
        assert not (self.components & rhs.components), "noise components not independent"
        self.components |= rhs.components
        self.noise_level_squared += rhs.noise_level_squared
        if self.noise_level_squared > max_noise_level_squared:
            raise NoiseTooBig(f"NoiseTooBig: {self.noise_level_squared} > {max_noise_level_squared}")


NOMINAL = 1


class BitCt:
    """Ciphertext of one bit under the big (GLWE) key — reference shortint_woppbs_1bit.rs:28-32, :86-122."""
    __slots__ = ("ct", "noise_level", "context")

    def __init__(self, ct, noise_level, context):
        self.ct, self.noise_level, self.context = ct, noise_level, context

    @classmethod
    def fresh(cls, ct, context):
        return cls.with_noise_level(ct, NOMINAL, context)

    @classmethod
    def with_noise_level(cls, ct, noise_level_squared, context):
        return cls(ct, NoiseLevelWithComponents.with_noise_level(noise_level_squared, context.next_ct_id()), context)

    @classmethod
    def trivial(cls, bit, context):
        ct = np.zeros(context.params.big_lwe_size, dtype=np.uint64)
        ct[-1] = encode_bit(bit)
        return cls(ct, NoiseLevelWithComponents.trivial(), context)

    def clone(self):
        return BitCt(self.ct.copy(), NoiseLevelWithComponents(self.noise_level.noise_level_squared, set(self.noise_level.components)), self.context)

    def __ixor__(self, rhs):
        """BitXorAssign (:134-142): lwe_ciphertext_add_assign + noise bookkeeping.  Element-wise wrapping add of 2049 words;
        batched XORs of whole states go through FheContext.lwe_add_batch / the fused AES path instead."""
        self.noise_level.add_assign(rhs.noise_level, self.context.params.max_noise_level_squared)
        self.ct = self.ct + rhs.ct
        return self

    def __xor__(self, rhs):
        out = self.clone()
        out ^= rhs
        return out


class NoiseContext:
    """The host-only part of FheContext: parameters + the ciphertext-id counter (reference :171, :175-178).  A ClientKey
    without a server context hands this to the BitCts it creates so that XOR bookkeeping works on the client alone."""

    def __init__(self, params):
        self.params = params if isinstance(params, Params) else params_preset(params)
        self._ct_counter = itertools.count()
        self._id_lock = threading.Lock()

    def next_ct_id(self):
        with self._id_lock:
            return next(self._ct_counter)

    def trivial(self, bit):
        return BitCt.trivial(bit, self)


_ctx_tokens = itertools.count(1)


class FheContext(NoiseContext):
    """Server-side context — reference FheContext (shortint_woppbs_1bit.rs:166-172): evaluation keys + parameters +
    ciphertext-id counter.  The keys live in HBM of one B200."""

    def __init__(self, params, device=0, stream=None):
        self.L = load_library()
        self.params = params if isinstance(params, Params) else params_preset(params)
        self.device = device
        self.h = self.L.tac_ctx_create(C.byref(self.params), device)
        if not self.h:
            raise RuntimeError("tac_ctx_create failed: " + (self.L.tac_last_error(None) or b"").decode())
        if stream is not None:
            self._check(self.L.tac_ctx_set_stream(self.h, C.c_void_p(stream)))
        self._token = next(_ctx_tokens)
        self._ct_counter = itertools.count()
        self._id_lock = threading.Lock()

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.L.tac_ctx_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # -- plumbing
    def last_error(self):
        return (self.L.tac_last_error(self.h) or b"").decode()

    def _check(self, rc):
        if rc == TAC_ERR_NOISE:
            raise NoiseTooBig(self.last_error())
        if rc != 0:
            raise RuntimeError(f"tfhe_aes_cuda error {rc}: {self.last_error()}")

    @classmethod
    def generate_keys(cls, pid, seed=None, device=0, stream=None):
        """generate_keys_sqrd_lvl_{1,4,64,256} (:229-243): returns (ClientKey, FheContext) with the keys uploaded."""
        ck = ClientKey(pid, seed).gen_eval_keys()
        ctx = cls(ck.params, device, stream)
        ctx.upload_keys(ck)
        ck.context = ctx
        return ck, ctx

    def upload_keys(self, client_key):
        bsk, ksk, pf = client_key.bsk, client_key.ksk, client_key.pfpksk
        self._check(self.L.tac_ctx_upload_keys(self.h, bsk.ctypes.data, ksk.ctypes.data, pf.ctypes.data))

    def load_keys(self, path):
        """evaluation keys from a wire file written by ClientKey.save_keys or by a tfhe-rs process (INTEGRATION.md)"""
        self._check(self.L.tac_ctx_load_keys(self.h, os.fsencode(path)))

    def alloc_keys(self):
        self._check(self.L.tac_ctx_alloc_keys(self.h))

    def key_buffer(self, which):
        ptr, nbytes = C.c_void_p(), C.c_size_t()
        self._check(self.L.tac_ctx_key_buffer(self.h, which, C.byref(ptr), C.byref(nbytes)))
        return ptr.value, nbytes.value

    def keys_ready(self):
        self._check(self.L.tac_ctx_keys_ready(self.h))

    def sync(self):
        self._check(self.L.tac_ctx_sync(self.h))

    def set_profiling(self, on=True):
        self._check(self.L.tac_ctx_set_profiling(self.h, int(on)))

    def stage_times(self):
        """summed per-stage device ms since the last call, plus the number of pipeline passes (= PBS kernel launches)"""
        arr, n = (C.c_float * 5)(), C.c_int()
        self._check(self.L.tac_ctx_stage_times(self.h, arr, C.byref(n)))
        d = dict(zip(("keyswitch", "pbs", "pfks", "ggsw_fft", "vertical_packing"), [float(x) for x in arr]))
        d["passes"] = n.value
        return d

    def fp64_peak_tflops(self):
        v = C.c_double()
        self._check(self.L.tac_bench_fp64_peak(self.h, C.byref(v)))
        return v.value

    def launch_count(self):
        return int(self.L.tac_ctx_launch_count(self.h))

    # -- the model API (ContextT::trivial, reference src/tfhe.rs:19-24, is inherited from NoiseContext)
    def generate_lookup_table(self, input_bits, output_bits, f):
        """reference :274-289"""
        return LookupTable(generate_multivariate_luts(input_bits, output_bits, self.params.polynomial_size, f), input_bits, output_bits)

    def circuit_bootstrap(self, bits, lut):
        """reference :292-336 — bits: list of BitCt; returns list of BitCt with noise level NOMINAL · len(bits)."""
        assert len(bits) == lut.input_bits
        arr = np.stack([b.ct for b in bits])[None]
        out = self.circuit_bootstrap_batch(arr, lut)[0]
        level = NOMINAL * len(bits)
        return [BitCt.with_noise_level(out[i].copy(), level, self) for i in range(lut.output_bits)]

    def circuit_bootstrap_coalesced(self, bits, lut):
        """circuit_bootstrap for callers that arrive from many threads (the reference's rayon pattern): concurrent calls
        are merged into one batched GPU pass (tac_wopbs_coalesced)."""
        assert len(bits) == lut.input_bits
        a = np.ascontiguousarray(np.stack([b.ct for b in bits]), dtype=np.uint64)
        out = np.empty((lut.output_bits, self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_wopbs_coalesced(self.h, lut.device_id(self), 1, a.ctypes.data, out.ctypes.data))
        level = NOMINAL * len(bits)
        return [BitCt.with_noise_level(out[i].copy(), level, self) for i in range(lut.output_bits)]

    def set_coalescing(self, window_us=200, max_batch=4096):
        self._check(self.L.tac_ctx_set_coalescing(self.h, window_us, max_batch))

    def coalescing_stats(self):
        r, p = C.c_uint64(), C.c_uint64()
        self._check(self.L.tac_ctx_coalescing_stats(self.h, C.byref(r), C.byref(p)))
        return {"requests": r.value, "passes": p.value}

    def circuit_bootstrap_batch(self, in_cts, lut):
        """batched raw form: in [batch][n_in][big+1] → out [batch][n_out][big+1] (host arrays)."""
        a = np.ascontiguousarray(in_cts, dtype=np.uint64)
        assert a.ndim == 3 and a.shape[1] == lut.input_bits and a.shape[2] == self.params.big_lwe_size
        out = np.empty((a.shape[0], lut.output_bits, self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_wopbs_batch(self.h, lut.device_id(self), a.shape[0], a.ctypes.data, out.ctypes.data))
        return out

    def lwe_add_batch(self, a, b):
        a = np.array(a, dtype=np.uint64, copy=True)
        b = np.ascontiguousarray(b, dtype=np.uint64)
        assert a.shape == b.shape
        n = a.size // self.params.big_lwe_size
        self._check(self.L.tac_lwe_add_batch(self.h, a.ctypes.data, b.ctypes.data, n))
        return a

    # -- fused AES (state resident on the device)
    def aes_set_key_schedule(self, key_sched):
        ks = np.ascontiguousarray(key_sched, dtype=np.uint64)
        assert ks.size == 44 * 32 * self.params.big_lwe_size
        self._check(self.L.tac_aes_set_key_schedule(self.h, ks.ctypes.data))

    def aes_key_schedule(self, key_bits):
        kb = np.ascontiguousarray(key_bits, dtype=np.uint64)
        assert kb.size == 128 * self.params.big_lwe_size
        out = np.empty((44, 4, 8, self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_aes_key_schedule(self.h, kb.ctypes.data, out.ctypes.data))
        return out

    def _aes_blocks(self, fn, blocks, rounds, in_noise_sq):
        b = np.ascontiguousarray(blocks, dtype=np.uint64).reshape(-1, 16, 8, self.params.big_lwe_size)
        out = np.empty_like(b)
        self._check(fn(self.h, b.shape[0], rounds, in_noise_sq, b.ctypes.data, out.ctypes.data))
        return out

    def aes_encrypt_blocks(self, blocks, rounds=10, in_noise_sq=1):
        return self._aes_blocks(self.L.tac_aes_encrypt_blocks, blocks, rounds, in_noise_sq)

    def aes_encrypt_blocks_dev(self, n_blocks, in_ptr, out_ptr, rounds=10, in_noise_sq=1):
        self._check(self.L.tac_aes_encrypt_blocks_dev(self.h, n_blocks, rounds, in_noise_sq, C.c_void_p(in_ptr), C.c_void_p(out_ptr)))

    # -- AES over public blocks: AES-CTR keystream and transciphering
    def _aes_public_blocks(self, fn, blocks, rounds, xor, dev=False, out_ptr=None):
        """fn on public blocks [n][16] with optional XOR bytes [n][16]: into device memory out_ptr (dev), else into the
        returned host array"""
        b = _public_blocks(blocks)
        x = None
        if xor is not None:
            x = _public_blocks(xor)
            if x.shape != b.shape:
                raise ValueError("xor must hold one 16-byte row per block")
        out = None if dev else np.empty((b.shape[0], 16, 8, self.params.big_lwe_size), dtype=np.uint64)
        self._check(fn(self.h, b.shape[0], rounds, b.ctypes.data, None if x is None else x.ctypes.data,
                       C.c_void_p(out_ptr) if dev else out.ctypes.data))
        return out

    def aes_encrypt_public_blocks(self, blocks, rounds=10, xor=None):
        """AES of public 16-byte blocks under the device key schedule; xor: optional public bytes [n][16] XORed into the
        output.  Returns [n][16][8][big+1] bit ciphertexts (squared noise level 9)."""
        return self._aes_public_blocks(self.L.tac_aes_encrypt_public_blocks, blocks, rounds, xor)

    def aes_encrypt_public_blocks_dev(self, blocks, out_ptr, rounds=10, xor=None):
        """the same into device memory out_ptr ([n][16][8][big+1] words), enqueued on the context's stream"""
        self._aes_public_blocks(self.L.tac_aes_encrypt_public_blocks_dev, blocks, rounds, xor, dev=True, out_ptr=out_ptr)

    def aes_ctr_keystream(self, iv, first_ctr, n_blocks):
        """FHE encryptions of the AES-CTR keystream blocks AES(k, iv ‖ BE64(first_ctr + i)): [n_blocks][16][8][big+1]"""
        return self.aes_encrypt_public_blocks(ctr_blocks(iv, first_ctr, n_blocks))

    def aes_ctr_transcipher(self, iv, first_ctr, data):
        """Transciphering: `data` is an AES-CTR ciphertext under the FHE-encrypted key (nonce iv ‖ BE64(first_ctr)); returns
        FHE encryptions of its plaintext bits, [len(data)][8][big+1]."""
        data = bytes(data)
        n = (len(data) + 15) // 16
        padded = data + bytes(16 * n - len(data))
        out = self.aes_encrypt_public_blocks(ctr_blocks(iv, first_ctr, n), xor=padded)
        return out.reshape(16 * n, 8, self.params.big_lwe_size)[:len(data)]

    # -- AES decryption (equivalent inverse cipher) and AES-ECB / AES-CBC transciphering
    def aes_inv_key_schedule(self):
        """derive the inverse key schedule dk on the device from the resident key schedule; returns it, [44][4][8][big+1].
        It stays in use until the key schedule changes (aes_set_key_schedule / aes_key_schedule make it stale)."""
        out = np.empty((44, 4, 8, self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_aes_inv_key_schedule(self.h, out.ctypes.data))
        return out

    def aes_set_inv_key_schedule(self, inv_key_sched):
        dk = np.ascontiguousarray(inv_key_sched, dtype=np.uint64)
        assert dk.size == 44 * 32 * self.params.big_lwe_size
        self._check(self.L.tac_aes_set_inv_key_schedule(self.h, dk.ctypes.data))

    def aes_decrypt_blocks(self, blocks, rounds=10, in_noise_sq=1):
        """AES decryption of FHE-encrypted blocks [n][16][8][big+1] under the resident inverse key schedule"""
        return self._aes_blocks(self.L.tac_aes_decrypt_blocks, blocks, rounds, in_noise_sq)

    def aes_decrypt_blocks_dev(self, n_blocks, in_ptr, out_ptr, rounds=10, in_noise_sq=1):
        self._check(self.L.tac_aes_decrypt_blocks_dev(self.h, n_blocks, rounds, in_noise_sq, C.c_void_p(in_ptr), C.c_void_p(out_ptr)))

    def aes_decrypt_public_blocks(self, blocks, rounds=10, xor=None):
        """AES decryption of public 16-byte ciphertext blocks; xor: optional public bytes [n][16] XORed into the output.
        Returns [n][16][8][big+1] bit ciphertexts (squared noise level 9)."""
        return self._aes_public_blocks(self.L.tac_aes_decrypt_public_blocks, blocks, rounds, xor)

    def aes_decrypt_public_blocks_dev(self, blocks, out_ptr, rounds=10, xor=None):
        """the same into device memory out_ptr ([n][16][8][big+1] words), enqueued on the context's stream"""
        self._aes_public_blocks(self.L.tac_aes_decrypt_public_blocks_dev, blocks, rounds, xor, dev=True, out_ptr=out_ptr)

    @staticmethod
    def _whole_blocks(data):
        data = bytes(data)
        if len(data) % 16:
            raise ValueError("AES-ECB / AES-CBC ciphertexts are whole 16-byte blocks")
        return data

    def aes_ecb_transcipher(self, data):
        """Transciphering: `data` is an AES-ECB ciphertext under the FHE-encrypted key; returns FHE encryptions of its
        (padded) plaintext bits, [len(data)][8][big+1].  Removing padding is the caller's business."""
        data = self._whole_blocks(data)
        return self.aes_decrypt_public_blocks(data).reshape(len(data), 8, self.params.big_lwe_size)

    def aes_cbc_transcipher(self, iv, data):
        """Transciphering: `data` is an AES-CBC ciphertext under the FHE-encrypted key with the 16-byte `iv`;
        P_i = AES^-1(C_i) xor C_{i-1}, C_{-1} = iv.  Returns FHE encryptions of the (padded) plaintext bits, [len(data)][8][big+1]."""
        iv, data = bytes(iv), self._whole_blocks(data)
        if len(iv) != 16:
            raise ValueError("iv must be 16 bytes")
        out = self.aes_decrypt_public_blocks(data, xor=(iv + data[:-16]) if data else None)
        return out.reshape(len(data), 8, self.params.big_lwe_size)

    # -- AES under many keys: a resident table of key schedules, one call over blocks of many keys
    def aes_key_table(self, keys_bits):
        """batched key expansion of K FHE-encrypted keys [K][128][big+1] (K >= 1); the result becomes the resident key
        table and is returned, [K][44][4][8][big+1].  Entry k equals aes_key_schedule of key k.  The single key schedule
        is left as it is; the inverse table becomes stale."""
        kb = np.ascontiguousarray(keys_bits, dtype=np.uint64)
        L1 = self.params.big_lwe_size
        if kb.size == 0 or kb.size % (128 * L1):
            raise ValueError("keys_bits must hold [K][128][big+1] words, K >= 1")
        K = kb.size // (128 * L1)
        out = np.empty((K, 44, 4, 8, L1), dtype=np.uint64)
        self._n_keys = 0
        self._check(self.L.tac_aes_key_table(self.h, K, kb.ctypes.data, out.ctypes.data))
        self._n_keys = K
        return out

    def aes_set_key_table(self, key_scheds):
        """make K expanded keys [K][44][4][8][big+1] the resident key table; the inverse table becomes stale"""
        ks = np.ascontiguousarray(key_scheds, dtype=np.uint64)
        per = 44 * 32 * self.params.big_lwe_size
        if ks.size == 0 or ks.size % per:
            raise ValueError("key_scheds must hold [K][44][4][8][big+1] words, K >= 1")
        self._n_keys = 0
        self._check(self.L.tac_aes_set_key_table(self.h, ks.size // per, ks.ctypes.data))
        self._n_keys = ks.size // per

    def aes_inv_key_table(self):
        """derive the inverse key schedule of every entry of the resident key table; returns them, [K][44][4][8][big+1]"""
        out = np.empty((max(self.n_keys, 1), 44, 4, 8, self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_aes_inv_key_table(self.h, out.ctypes.data))
        return out

    def aes_set_inv_key_table(self, inv_key_scheds):
        """make given inverse schedules [K][44][4][8][big+1] resident, K of the resident key table"""
        dk = np.ascontiguousarray(inv_key_scheds, dtype=np.uint64)
        if dk.size != self.n_keys * 44 * 32 * self.params.big_lwe_size:
            raise ValueError(f"inverse key schedules must match the resident key table of {self.n_keys} keys")
        self._check(self.L.tac_aes_set_inv_key_table(self.h, dk.ctypes.data))

    @property
    def n_keys(self):
        """entries of the resident key table (0: none)"""
        return getattr(self, "_n_keys", 0)

    def _aes_blocks_keyed(self, fn, blocks, key_index, rounds, in_noise_sq):
        b = np.ascontiguousarray(blocks, dtype=np.uint64).reshape(-1, 16, 8, self.params.big_lwe_size)
        k = _key_index(key_index, b.shape[0], self.n_keys)
        out = np.empty_like(b)
        self._check(fn(self.h, b.shape[0], rounds, in_noise_sq, k.ctypes.data, b.ctypes.data, out.ctypes.data))
        return out

    def _aes_blocks_keyed_dev(self, fn, n_blocks, key_index, in_ptr, out_ptr, rounds, in_noise_sq):
        k = _key_index(key_index, n_blocks, self.n_keys)
        self._check(fn(self.h, n_blocks, rounds, in_noise_sq, k.ctypes.data, C.c_void_p(in_ptr), C.c_void_p(out_ptr)))

    def aes_encrypt_blocks_keyed(self, blocks, key_index, rounds=10, in_noise_sq=1):
        """aes_encrypt_blocks with block b under key table entry key_index[b]"""
        return self._aes_blocks_keyed(self.L.tac_aes_encrypt_blocks_keyed, blocks, key_index, rounds, in_noise_sq)

    def aes_encrypt_blocks_keyed_dev(self, n_blocks, key_index, in_ptr, out_ptr, rounds=10, in_noise_sq=1):
        self._aes_blocks_keyed_dev(self.L.tac_aes_encrypt_blocks_keyed_dev, n_blocks, key_index, in_ptr, out_ptr, rounds, in_noise_sq)

    def aes_decrypt_blocks_keyed(self, blocks, key_index, rounds=10, in_noise_sq=1):
        """aes_decrypt_blocks with block b under inverse table entry key_index[b]"""
        return self._aes_blocks_keyed(self.L.tac_aes_decrypt_blocks_keyed, blocks, key_index, rounds, in_noise_sq)

    def aes_decrypt_blocks_keyed_dev(self, n_blocks, key_index, in_ptr, out_ptr, rounds=10, in_noise_sq=1):
        self._aes_blocks_keyed_dev(self.L.tac_aes_decrypt_blocks_keyed_dev, n_blocks, key_index, in_ptr, out_ptr, rounds, in_noise_sq)

    def _aes_public_blocks_keyed(self, fn, blocks, key_index, rounds, xor, dev=False, out_ptr=None):
        b = _public_blocks(blocks)
        k = _key_index(key_index, b.shape[0], self.n_keys)
        return self._aes_public_blocks(lambda h, n, r, bp, xp, op: fn(h, n, r, k.ctypes.data, bp, xp, op), b, rounds, xor, dev, out_ptr)

    def aes_encrypt_public_blocks_keyed(self, blocks, key_index, rounds=10, xor=None):
        """aes_encrypt_public_blocks with block b under key table entry key_index[b]"""
        return self._aes_public_blocks_keyed(self.L.tac_aes_encrypt_public_blocks_keyed, blocks, key_index, rounds, xor)

    def aes_encrypt_public_blocks_keyed_dev(self, blocks, key_index, out_ptr, rounds=10, xor=None):
        self._aes_public_blocks_keyed(self.L.tac_aes_encrypt_public_blocks_keyed_dev, blocks, key_index, rounds, xor, dev=True, out_ptr=out_ptr)

    def aes_decrypt_public_blocks_keyed(self, blocks, key_index, rounds=10, xor=None):
        """aes_decrypt_public_blocks with block b under inverse table entry key_index[b]"""
        return self._aes_public_blocks_keyed(self.L.tac_aes_decrypt_public_blocks_keyed, blocks, key_index, rounds, xor)

    def aes_decrypt_public_blocks_keyed_dev(self, blocks, key_index, out_ptr, rounds=10, xor=None):
        self._aes_public_blocks_keyed(self.L.tac_aes_decrypt_public_blocks_keyed_dev, blocks, key_index, rounds, xor, dev=True, out_ptr=out_ptr)

    def aes_ctr_transcipher_many(self, messages):
        """aes_ctr_transcipher for many senders in one call: messages = [(key_index, iv, first_ctr, data)], each an AES-CTR
        ciphertext under key table entry key_index.  Returns one array per message, [len(data)][8][big+1]."""
        blocks, xor, kidx, sizes = [], [], [], []
        for key_index, iv, first_ctr, data in messages:
            data = bytes(data)
            n = (len(data) + 15) // 16
            blocks.append(ctr_blocks(iv, first_ctr, n))
            xor.append(data + bytes(16 * n - len(data)))
            kidx += [key_index] * n
            sizes.append(len(data))
        k = _key_index(kidx, len(kidx), self.n_keys)
        if not sizes:
            return []
        out = self.aes_encrypt_public_blocks_keyed(np.concatenate(blocks), k, xor=b"".join(xor))
        return self._split_messages(out, sizes)

    def aes_cbc_transcipher_many(self, messages):
        """aes_cbc_transcipher for many senders in one call: messages = [(key_index, iv, data)], each an AES-CBC ciphertext
        under key table entry key_index.  Returns one array per message, [len(data)][8][big+1]."""
        blocks, xor, kidx, sizes = [], [], [], []
        for key_index, iv, data in messages:
            iv, data = bytes(iv), self._whole_blocks(data)
            if len(iv) != 16:
                raise ValueError("iv must be 16 bytes")
            blocks.append(data)
            xor.append((iv + data[:-16]) if data else b"")
            kidx += [key_index] * (len(data) // 16)
            sizes.append(len(data))
        k = _key_index(kidx, len(kidx), self.n_keys)
        if not sizes:
            return []
        out = self.aes_decrypt_public_blocks_keyed(b"".join(blocks), k, xor=b"".join(xor))
        return self._split_messages(out, sizes)

    # -- AES-CCM transciphering with the tag checked under FHE
    def aes_ccm_transcipher(self, nonce, data, tag_len=16, aad=b""):
        """Transciphering of one AES-CCM record under the resident key schedule: `data` = C ‖ U is what AES-CCM encryption
        of (nonce, P, aad) returns, with a tag of tag_len bytes.  Returns (FHE encryptions of the plaintext bits
        [len(data) − tag_len][8][big+1], an encrypted validity bit [big+1]: 1 exactly when the tag is genuine).  The
        plaintext comes back whatever the tag; acting on the validity bit is the caller's business."""
        return self._aes_records(self.L.tac_aes_ccm_transcipher, _ccm_messages, [(nonce, data, tag_len, aad)], None)[0]

    def aes_ccm_transcipher_many(self, messages):
        """aes_ccm_transcipher for many senders in one call: messages = [(key_index, nonce, data, tag_len, aad)], each
        under key table entry key_index.  Returns one (plaintext bits, validity bit) pair per message."""
        messages = list(messages)
        k = _key_index([m[0] for m in messages], len(messages), self.n_keys)
        return self._aes_records(self.L.tac_aes_ccm_transcipher, _ccm_messages, [m[1:] for m in messages], k)

    def _aes_records(self, fn, build, messages, key_index):
        """fn (tac_aes_ccm_transcipher / tac_aes_gcm_transcipher) over the records that build (_ccm_messages /
        _gcm_messages) makes of messages; one (plaintext bits, validity bit) pair per record"""
        msgs, keep, sizes = build(messages)
        if not sizes:
            return []
        L1 = self.params.big_lwe_size
        pt = np.empty((sum(sizes), 8, L1), dtype=np.uint64)
        valid = np.empty((len(sizes), L1), dtype=np.uint64)
        self._check(fn(self.h, len(sizes), None if key_index is None else key_index.ctypes.data, msgs, pt.ctypes.data, valid.ctypes.data))
        offs = np.cumsum([0] + sizes)
        return [(pt[offs[i]:offs[i + 1]], valid[i]) for i in range(len(sizes))]

    # -- AES-GCM transciphering with the tag checked under FHE
    def aes_gcm_hash_key(self, depth=8):
        """GHASH key table of the resident key schedule: H = E_K(0) and its powers H^1..H^depth, returned as
        [depth][128][big+1] (bit order of the state).  It stays valid until the key schedule changes."""
        depth = _gcm_depth(depth)
        out = np.empty((depth, 128, self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_aes_gcm_hash_key(self.h, depth, out.ctypes.data))
        return out

    def aes_gcm_hash_key_table(self, depth=8):
        """GHASH key tables of every entry of the resident key table, [K][depth][128][big+1]; valid until the key table
        changes"""
        depth = _gcm_depth(depth)
        out = np.empty((max(self.n_keys, 1), depth, 128, self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_aes_gcm_hash_key_table(self.h, depth, out.ctypes.data))
        return out

    def aes_gcm_transcipher(self, iv, data, tag_len=16, aad=b""):
        """Transciphering of one AES-GCM record under the resident key schedule and its GHASH key table: `data` = C ‖ T is
        what AES-GCM encryption of (iv, P, aad) returns.  Returns (FHE encryptions of the plaintext bits
        [len(data) − tag_len][8][big+1], an encrypted validity bit [big+1]: 1 exactly when the tag is genuine)."""
        return self._aes_records(self.L.tac_aes_gcm_transcipher, _gcm_messages, [(iv, data, tag_len, aad)], None)[0]

    def aes_gcm_transcipher_many(self, messages):
        """aes_gcm_transcipher for many senders in one call: messages = [(key_index, iv, data, tag_len, aad)], each under
        key table entry key_index.  Returns one (plaintext bits, validity bit) pair per record."""
        messages = list(messages)
        k = _key_index([m[0] for m in messages], len(messages), self.n_keys)
        return self._aes_records(self.L.tac_aes_gcm_transcipher, _gcm_messages, [m[1:] for m in messages], k)

    def gf128_mul(self, a, b):
        """encrypted products a·b in GF(2^128) (GCM's field and bit order): a, b [n][128][big+1] → [n][128][big+1], output
        bits at squared noise 1"""
        L1 = self.params.big_lwe_size
        x = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 128, L1)
        y = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, 128, L1)
        if x.shape != y.shape:
            raise ValueError("gf128_mul: operands of different counts")
        out = np.empty_like(x)
        self._check(self.L.tac_gf128_mul(self.h, x.shape[0], x.reshape(-1), y.reshape(-1), out.reshape(-1)))
        return out

    def _split_messages(self, out, sizes):
        """[n][16][8][big+1] of whole blocks → one [size][8][big+1] array per message (each padded to whole blocks)"""
        flat = out.reshape(-1, 8, self.params.big_lwe_size)
        res, off = [], 0
        for n in sizes:
            res.append(flat[off:off + n])
            off += 16 * ((n + 15) // 16)
        return res

    def aes_key_schedule_buffer(self):
        ptr, nbytes = C.c_void_p(), C.c_size_t()
        self._check(self.L.tac_aes_key_schedule_buffer(self.h, C.byref(ptr), C.byref(nbytes)))
        return ptr.value, nbytes.value

    # -- single stages
    def stage_keyswitch(self, cts):
        a = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, self.params.big_lwe_size)
        out = np.empty((a.shape[0], self.params.lwe_dimension + 1), dtype=np.uint64)
        self._check(self.L.tac_stage_keyswitch(self.h, a.shape[0], a, out))
        return out

    def extract_bits(self, cts, delta_log, n_bits):
        """WopbsKey::extract_bits: [n][big+1] → [n][n_bits][small+1], most significant extracted bit first"""
        a = np.ascontiguousarray(cts, dtype=np.uint64).reshape(-1, self.params.big_lwe_size)
        out = np.empty((a.shape[0], n_bits, self.params.lwe_dimension + 1), dtype=np.uint64)
        self._check(self.L.tac_extract_bits(self.h, delta_log, n_bits, a.shape[0], a, out.reshape(-1)))
        return out

    def stage_pbs(self, small):
        a = np.ascontiguousarray(small, dtype=np.uint64).reshape(-1, self.params.lwe_dimension + 1)
        out = np.empty((a.shape[0], self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_stage_pbs(self.h, a.shape[0], a, out))
        return out

    def stage_pfks(self, bigs):
        a = np.ascontiguousarray(bigs, dtype=np.uint64).reshape(-1, self.params.big_lwe_size)
        G = self.params.glwe_dimension + 1
        out = np.empty((a.shape[0], G, G * self.params.polynomial_size), dtype=np.uint64)
        self._check(self.L.tac_stage_pfks(self.h, a.shape[0], a, out))
        return out

    def stage_vertical_packing(self, ggsw_std, lut):
        G, N = self.params.glwe_dimension + 1, self.params.polynomial_size
        g = np.ascontiguousarray(ggsw_std, dtype=np.uint64).reshape(-1, lut.input_bits, self.params.cbs_level, G, G * N)
        out = np.empty((g.shape[0], lut.output_bits, self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_stage_vertical_packing(self.h, lut.device_id(self), g.shape[0], g.reshape(-1), out.reshape(-1)))
        return out

    def stage_poly_fft(self, polys):
        """fill_with_forward_fourier of torus polynomials [n][N] → complex [n][N/2] in slot order (see fft_slot_frequencies)"""
        N = self.params.polynomial_size
        a = np.ascontiguousarray(polys, dtype=np.uint64).reshape(-1, N)
        out = np.empty((a.shape[0], N // 2, 2), dtype=np.float64)
        self._check(self.L.tac_stage_poly_fft(self.h, a.shape[0], a.reshape(-1), out.reshape(-1)))
        return out[..., 0] + 1j * out[..., 1]

    def fft_slot_frequencies(self):
        f = np.empty(self.params.polynomial_size // 2, dtype=np.int32)
        assert self.L.tac_fft_slot_frequencies(self.params.polynomial_size, f) == 0
        return f

    def stage_sample_extract(self, glwes):
        G, N = self.params.glwe_dimension + 1, self.params.polynomial_size
        g = np.ascontiguousarray(glwes, dtype=np.uint64).reshape(-1, G * N)
        out = np.empty((g.shape[0], self.params.big_lwe_size), dtype=np.uint64)
        self._check(self.L.tac_stage_sample_extract(self.h, g.shape[0], g.reshape(-1), out.reshape(-1)))
        return out

    def stage_cmux_rotate(self, ggsw_std, levels, base_log, acc, rot):
        G, N = self.params.glwe_dimension + 1, self.params.polynomial_size
        a = np.array(acc, dtype=np.uint64, copy=True).reshape(-1, G * N)
        r = np.ascontiguousarray(rot, dtype=np.int32)
        g = np.ascontiguousarray(ggsw_std, dtype=np.uint64).reshape(-1)
        assert g.size == levels * G * G * N and r.size == a.shape[0]
        self._check(self.L.tac_stage_cmux_rotate(self.h, levels, base_log, g, a.shape[0], r, a.reshape(-1)))
        return a
