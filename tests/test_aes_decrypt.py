"""AES-128 decryption with the equivalent inverse cipher (FIPS-197 §5.3.5) and AES-ECB / AES-CBC transciphering.

CPU: this file's clear inverse cipher against the oracle's forward cipher and against `cryptography`, and the inverse
sharing plan against a brute-force restatement of its rule.  B200: FIPS-197 C.1 under a derived and an uploaded inverse
key schedule, round trips through the encryption path, word-for-word identity of the public-block path with the
encrypted-block path on trivial ciphertexts, CBC / ECB transciphering, and the error paths."""
import numpy as np
import pytest

from test_oracle_golden import CLI_IV, CLI_KEY

TAC_ERR_ARG, TAC_ERR_STATE = -2, -3

FIPS_KEY = bytes(range(16))
FIPS_PT = bytes.fromhex("00112233445566778899aabbccddeeff")
FIPS_CT = bytes.fromhex("69c4e0d86a7b0430d8cdb78070b4c55a")


# ---------------------------------------------------------------------------------------------- clear reference
def _tables(ol):
    S = [ol.sbox(i) for i in range(256)]
    IS = [0] * 256
    for i, s in enumerate(S):
        IS[s] = i
    return S, IS


def inv_mix_column(ol, col):
    """col: 4 bytes (rows 0..3) → InvMixColumns, row r = Σ_r' coef[(r' − r) mod 4]·col[r'], coef = (14, 11, 13, 9)"""
    coef = (14, 11, 13, 9)
    out = []
    for r in range(4):
        v = 0
        for rr in range(4):
            v ^= ol.gf_256_mul(col[rr], coef[(rr - r) & 3])
        out.append(v)
    return out


def inv_mix_columns(ol, s):
    return [b for c in range(4) for b in inv_mix_column(ol, s[4 * c:4 * c + 4])]


def inv_shift_rows(s):
    """new[row][c] = old[row][(c − row) mod 4], byte index 4·col + row"""
    return [s[4 * ((c - r) & 3) + r] for c in range(4) for r in range(4)]


def plain_decrypt_block(ol, key, block, rounds=10):
    """straight inverse cipher (FIPS-197 §5.3) of ol.plain_encrypt_block(key, ·, rounds), whose final round adds rk10 for
    every `rounds`"""
    _, IS = _tables(ol)
    ek = list(ol.plain_key_schedule(key))
    rk = lambda i: ek[16 * i:16 * i + 16]
    s = [a ^ b for a, b in zip(block, rk(10))]
    s = [IS[b] for b in inv_shift_rows(s)]
    for rd in range(rounds - 1, 0, -1):
        s = [a ^ b for a, b in zip(s, rk(rd))]
        s = inv_mix_columns(ol, s)
        s = [IS[b] for b in inv_shift_rows(s)]
    return bytes(a ^ b for a, b in zip(s, rk(0)))


def clear_inv_key_schedule(ol, key):
    """dk of the equivalent inverse cipher: w[0..3], InvMixColumns(w[4rd..4rd+3]) for rd = 1..9, w[40..43] (176 bytes)"""
    ek = list(ol.plain_key_schedule(key))
    dk = ek[:16]
    for rd in range(1, 10):
        dk += inv_mix_columns(ol, ek[16 * rd:16 * rd + 16])
    return bytes(dk + ek[160:])


def equivalent_decrypt_block(ol, dk, block, rounds=10):
    """the device's round structure in the clear: s = in ⊕ dk[10]; rd = rounds−1 … 1: InvMixColumns(InvShiftRows(InvS(s))) ⊕ dk[rd]"""
    _, IS = _tables(ol)
    rk = lambda i: dk[16 * i:16 * i + 16]
    s = [a ^ b for a, b in zip(block, rk(10))]
    for rd in range(rounds - 1, 0, -1):
        s = [a ^ b for a, b in zip(inv_mix_columns(ol, inv_shift_rows([IS[b] for b in s])), rk(rd))]
    return bytes(a ^ b for a, b in zip(inv_shift_rows([IS[b] for b in s]), rk(0)))


def seeded_blocks(n, seed=7):
    raw = np.random.default_rng(seed).bytes(16 * n)
    return [raw[16 * i:16 * i + 16] for i in range(n)]


def test_inverse_cipher_inverts_reduced_rounds(ol):
    for rounds in range(1, 11):
        for b in seeded_blocks(4, seed=rounds):
            ct = ol.plain_encrypt_block(CLI_KEY, b, rounds)
            assert plain_decrypt_block(ol, CLI_KEY, ct, rounds) == b, rounds
            assert equivalent_decrypt_block(ol, clear_inv_key_schedule(ol, CLI_KEY), ct, rounds) == b, rounds


def test_inverse_cipher_matches_cryptography(ol):
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    blocks = seeded_blocks(8, seed=11)
    dec = Cipher(algorithms.AES(CLI_KEY), modes.ECB()).decryptor().update(b"".join(blocks))
    assert b"".join(plain_decrypt_block(ol, CLI_KEY, b) for b in blocks) == dec
    assert plain_decrypt_block(ol, FIPS_KEY, FIPS_CT) == FIPS_PT                       # FIPS-197 C.1


# ---------------------------------------------------------------------------------------------- the inverse plan (host only)
def dependence_sets(rounds, inverse):
    """D(1, j) = {j}, D(r+1, (row, c)) = U_{r'} D(r, 4((c ∓ r') mod 4) + r'): ShiftRows forward, InvShiftRows inverse"""
    sgn = -1 if inverse else 1
    D = [{j} for j in range(16)]
    out = [D]
    for _ in range(1, rounds):
        D = [set().union(*(D[4 * (((j >> 2) + sgn * rr) & 3) + rr] for rr in range(4))) for j in range(16)]
        out.append(D)
    return out


def brute_force_plan(blocks, rounds=10, inverse=True):
    blocks = [bytes(b) for b in blocks]
    return [sum(len({tuple(b[i] for i in sorted(D[j])) for b in blocks}) for j in range(16)) for D in dependence_sets(rounds, inverse)]


def test_inverse_dependence_runs_along_the_other_diagonal():
    D = dependence_sets(3, inverse=True)
    assert D[1][0] == {0, 13, 10, 7} and D[1][4] == {4, 1, 14, 11}
    assert all(d == set(range(16)) for d in D[2])
    assert D[1][0] != dependence_sets(2, inverse=False)[1][0]


def test_plan_inv_random_blocks(tac):
    blocks = seeded_blocks(64, seed=3)
    for rounds in (1, 2, 10):
        got = tac.aes_public_plan(blocks, rounds, decrypt=True)
        assert got == brute_force_plan(blocks, rounds)
    assert tac.aes_public_plan(blocks, decrypt=True)[1:] == [16 * 64] * 9


def test_plan_inv_shares_on_the_inverse_diagonals(tac):
    """two blocks that agree only on {0, 7, 10, 13}, the inputs of column 0 in round 2 of decryption: its 4 boxes are shared
    there, while encryption's round-2 column 0 ({0, 5, 10, 15}) shares nothing"""
    base = bytes(seeded_blocks(1, seed=5)[0])
    other = bytes(b if j in (0, 7, 10, 13) else b ^ 0x5A for j, b in enumerate(base))
    blocks = [base, other]
    assert tac.aes_public_plan(blocks, 2, decrypt=True) == brute_force_plan(blocks, 2) == [16 + 12, 16 + 12]
    assert tac.aes_public_plan(blocks, 2) == brute_force_plan(blocks, 2, inverse=False) == [16 + 12, 32]


def test_plan_inv_duplicates_share_in_every_round(tac):
    distinct = seeded_blocks(5, seed=9)
    blocks = distinct + distinct[:2]                                    # blocks 5, 6 repeat blocks 0, 1
    got = tac.aes_public_plan(blocks, decrypt=True)
    assert got == brute_force_plan(blocks)
    assert all(n <= 16 * 5 for n in got) and got[2:] == [16 * 5] * 8
    assert tac.aes_public_plan([bytes(16)] * 4, decrypt=True) == [16] * 10
    assert tac.aes_public_plan([], 10, decrypt=True) == [0] * 10


def test_plan_inv_argument_errors(tac):
    for rounds in (0, 11):
        with pytest.raises(ValueError):
            tac.aes_public_plan(seeded_blocks(2), rounds, decrypt=True)
    L = tac.load_library()
    boxes = np.zeros(10, dtype=np.int64)
    blk = np.zeros(16, dtype=np.uint8)
    assert L.tac_aes_public_plan_inv(-1, 10, blk.ctypes.data, boxes.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_public_plan_inv(1, 10, None, boxes.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_public_plan_inv(1, 10, blk.ctypes.data, None) == TAC_ERR_ARG
    assert L.tac_aes_public_plan_inv(0, 10, None, boxes.ctypes.data) == 0


def test_forward_plan_unchanged(tac):
    blocks = [CLI_IV + (1 + i).to_bytes(8, "big") for i in range(128)]
    assert tac.aes_public_plan(blocks) == [143, 524, 2048] + [2048] * 7
    assert tac.aes_public_plan(blocks, decrypt=True) == brute_force_plan(blocks)


def test_transcipher_arguments_need_whole_blocks(tac):
    """the Python checks run before any device call"""
    ctx = object.__new__(tac.FheContext)
    with pytest.raises(ValueError):
        ctx.aes_ecb_transcipher(b"\x00" * 17)
    with pytest.raises(ValueError):
        ctx.aes_cbc_transcipher(b"\x00" * 16, b"\x00" * 31)
    with pytest.raises(ValueError):
        ctx.aes_cbc_transcipher(b"\x00" * 8, b"\x00" * 32)


# ---------------------------------------------------------------------------------------------- the device path
def clear_key_schedule_cts(ck, ol, key):
    return ck.encrypt_bytes(bytes(ol.plain_key_schedule(key)), first_index=1 << 40)


def clear_inv_key_schedule_cts(ck, ol, key):
    return ck.encrypt_bytes(clear_inv_key_schedule(ol, key), first_index=1 << 41)


def with_clear_schedules(ck, ctx, ol, key=CLI_KEY):
    ctx.aes_set_key_schedule(clear_key_schedule_cts(ck, ol, key))
    ctx.aes_set_inv_key_schedule(clear_inv_key_schedule_cts(ck, ol, key))


def trivial_blocks(blocks, L1):
    """trivial encryptions (mask 0, body encode_bit) of public blocks: [n][16][8][L1]"""
    b = np.unpackbits(np.frombuffer(b"".join(blocks), dtype=np.uint8).reshape(-1, 16), axis=1).reshape(-1, 16, 8)
    out = np.zeros(b.shape + (L1,), dtype=np.uint64)
    out[..., -1] = b.astype(np.uint64) << np.uint64(63)
    return out


@pytest.mark.gpu
def test_fips197_c1_derived_inverse_key_schedule(gpu64, ol):
    ck, ctx = gpu64
    ctx.aes_key_schedule(ck.encrypt_bytes(FIPS_KEY, first_index=1 << 44))
    dk = ctx.aes_inv_key_schedule()
    assert ck.decrypt_bytes(dk.reshape(-1, ck.params.big_lwe_size)) == clear_inv_key_schedule(ol, FIPS_KEY)
    out = ctx.aes_decrypt_blocks(ck.encrypt_bytes(FIPS_CT, first_index=1 << 43))
    assert ck.decrypt_bytes(out[0]) == FIPS_PT


@pytest.mark.gpu
def test_fips197_c1_uploaded_inverse_key_schedule(gpu64, ol):
    ck, ctx = gpu64
    with_clear_schedules(ck, ctx, ol, FIPS_KEY)
    out = ctx.aes_decrypt_blocks(ck.encrypt_bytes(FIPS_CT, first_index=1 << 43))
    assert ck.decrypt_bytes(out[0]) == FIPS_PT
    assert ck.decrypt_bytes(ctx.aes_decrypt_public_blocks(FIPS_CT)[0]) == FIPS_PT


@pytest.mark.gpu
@pytest.mark.parametrize("rounds", [1, 2, 10])
def test_round_trip_through_encryption(gpu64, ol, rounds):
    ck, ctx = gpu64
    with_clear_schedules(ck, ctx, ol)
    blocks = seeded_blocks(3, seed=100 + rounds)
    cts = np.stack([ck.encrypt_bytes(b, first_index=(1 + i) * 128) for i, b in enumerate(blocks)])
    enc = ctx.aes_encrypt_blocks(cts, rounds=rounds)
    for i, b in enumerate(blocks):
        assert ck.decrypt_bytes(enc[i]) == ol.plain_encrypt_block(CLI_KEY, b, rounds)
    dec = ctx.aes_decrypt_blocks(enc, rounds=rounds, in_noise_sq=9)
    for i, b in enumerate(blocks):
        assert ck.decrypt_bytes(dec[i]) == b


def assert_bit_identical(ctx, blocks, rounds, xor=None):
    L1 = ctx.params.big_lwe_size
    pub = ctx.aes_decrypt_public_blocks(blocks, rounds=rounds, xor=xor)
    ref = ctx.aes_decrypt_blocks(trivial_blocks(blocks, L1), rounds=rounds, in_noise_sq=0)
    if xor is not None:
        ref = ref.copy()
        ref[..., -1] += trivial_blocks(xor, L1)[..., -1]
    assert pub.shape == ref.shape
    bad = np.flatnonzero((pub != ref).any(axis=-1))
    assert bad.size == 0, f"rounds={rounds}: {bad.size} output bits differ, first at {bad[:8].tolist()}"
    return pub


@pytest.mark.gpu
@pytest.mark.parametrize("rounds", [1, 2, 10])
def test_bit_identical_to_encrypted_path(gpu64, tac, ol, rounds):
    """ECB-like set: shares in rounds 1 and 2 and holds a duplicate block (shares in every round)"""
    ck, ctx = gpu64
    with_clear_schedules(ck, ctx, ol)
    base = seeded_blocks(1, seed=21)[0]
    blocks = [base[:15] + bytes([i]) for i in range(5)] + [base[:15] + b"\x02", bytes(range(16))]
    assert all(n < 16 * len(blocks) for n in tac.aes_public_plan(blocks, rounds, decrypt=True))
    pub = assert_bit_identical(ctx, blocks, rounds)
    assert np.array_equal(pub[2], pub[5])                        # identical public blocks: word-identical outputs
    for i, b in enumerate(blocks):
        assert ck.decrypt_bytes(pub[i]) == plain_decrypt_block(ol, CLI_KEY, b, rounds)


@pytest.mark.gpu
def test_bit_identical_130_blocks(gpu64, ol):
    """rounds 3+ bootstrap 16·130 = 2080 boxes, more than one pass of the pipeline (2048 boxes at the default max_cts)"""
    ck, ctx = gpu64
    with_clear_schedules(ck, ctx, ol)
    blocks = seeded_blocks(130, seed=130)
    xor = seeded_blocks(130, seed=131)
    pub = assert_bit_identical(ctx, blocks, 10, xor=xor)
    for i in (0, 57, 129):
        want = bytes(a ^ b for a, b in zip(plain_decrypt_block(ol, CLI_KEY, blocks[i]), xor[i]))
        assert ck.decrypt_bytes(pub[i]) == want


@pytest.mark.gpu
def test_cbc_transcipher(gpu64, ol):
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    ck, ctx = gpu64
    with_clear_schedules(ck, ctx, ol)
    iv = np.random.default_rng(2026).bytes(16)
    msg = b"AES-CBC in, FHE out: the server never sees it."
    msg += b"." * (48 - len(msg))
    ct = Cipher(algorithms.AES(CLI_KEY), modes.CBC(iv)).encryptor().update(msg)
    out = ctx.aes_cbc_transcipher(iv, ct)
    assert out.shape == (48, 8, ck.params.big_lwe_size)
    assert ck.decrypt_bytes(out) == msg


@pytest.mark.gpu
def test_ecb_transcipher_repeated_block(gpu64, tac, ol):
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    ck, ctx = gpu64
    with_clear_schedules(ck, ctx, ol)
    msg = b"sixteen byte blk" * 2 + b"and another one!"
    ct = Cipher(algorithms.AES(CLI_KEY), modes.ECB()).encryptor().update(msg)
    plan = tac.aes_public_plan(ct, decrypt=True)
    assert plan == brute_force_plan([ct[i:i + 16] for i in range(0, 48, 16)]) and plan[2:] == [32] * 8   # the repeat shares every round
    out = ctx.aes_ecb_transcipher(ct)
    assert out.shape == (48, 8, ck.params.big_lwe_size)
    assert ck.decrypt_bytes(out) == msg
    assert np.array_equal(out[:16], out[16:32])


@pytest.mark.gpu
def test_device_entry_points(gpu64, ol):
    import torch
    ck, ctx = gpu64
    with_clear_schedules(ck, ctx, ol)
    blocks = seeded_blocks(3, seed=33)
    L1 = ck.params.big_lwe_size
    out = torch.empty((3, 16, 8, L1), dtype=torch.int64, device="cuda:0")
    ctx.aes_decrypt_public_blocks_dev(blocks, out.data_ptr(), rounds=2, xor=blocks[::-1])
    ctx.sync()
    host = ctx.aes_decrypt_public_blocks(blocks, rounds=2, xor=blocks[::-1])
    assert np.array_equal(out.cpu().numpy().view(np.uint64), host)

    cts = np.stack([ck.encrypt_bytes(b, first_index=(1 + i) * 128) for i, b in enumerate(blocks)])
    in_dev = torch.from_numpy(cts.view(np.int64)).to("cuda:0")
    ctx.aes_decrypt_blocks_dev(3, in_dev.data_ptr(), out.data_ptr(), rounds=2)
    ctx.sync()
    host = ctx.aes_decrypt_blocks(cts, rounds=2)
    assert np.array_equal(out.cpu().numpy().view(np.uint64), host)


@pytest.mark.gpu
def test_argument_errors(gpu64, ol):
    ck, ctx = gpu64
    with_clear_schedules(ck, ctx, ol)
    L = ctx.L
    blk = np.zeros(16, dtype=np.uint8)
    out = np.zeros((1, 16, 8, ck.params.big_lwe_size), dtype=np.uint64)
    for n, rounds, ptr in ((-1, 10, blk.ctypes.data), (1, 0, blk.ctypes.data), (1, 11, blk.ctypes.data), (1, 10, None)):
        assert L.tac_aes_decrypt_public_blocks(ctx.h, n, rounds, ptr, None, out.ctypes.data) == TAC_ERR_ARG
        assert L.tac_aes_decrypt_public_blocks_dev(ctx.h, n, rounds, ptr, None, None) == TAC_ERR_ARG
    for n, rounds in ((-1, 10), (1, 0), (1, 11)):
        assert L.tac_aes_decrypt_blocks(ctx.h, n, rounds, 1, out.ctypes.data, out.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_set_inv_key_schedule(ctx.h, None) == TAC_ERR_ARG


@pytest.mark.gpu
def test_state_errors_and_noise_guard(tac):
    """a context that never held dk, a stale dk, and params_sqrd_lvl_4, which cannot hold the squared noise 32 of the
    InvMixColumns sums nor the 33 of a middle round: NoiseTooBig for the inverse key schedule and for decryption"""
    ck = tac.ClientKey(4, seed=1).gen_eval_keys()
    ctx = tac.FheContext(ck.params)
    ctx.upload_keys(ck)
    L1 = ck.params.big_lwe_size
    zeros = np.zeros((44, 4, 8, L1), dtype=np.uint64)
    ctx.aes_set_key_schedule(zeros)
    with pytest.raises(RuntimeError, match="tac_aes_inv_key_schedule"):
        ctx.aes_decrypt_public_blocks(seeded_blocks(1), rounds=2)
    with pytest.raises(tac.NoiseTooBig):
        ctx.aes_inv_key_schedule()
    ctx.aes_set_inv_key_schedule(zeros)
    with pytest.raises(tac.NoiseTooBig):
        ctx.aes_decrypt_public_blocks(seeded_blocks(1), rounds=2)
    with pytest.raises(tac.NoiseTooBig):
        ctx.aes_decrypt_blocks(np.zeros((1, 16, 8, L1), dtype=np.uint64), rounds=2)
    ctx.aes_set_key_schedule(zeros)                                 # a new encryption schedule: dk is stale
    blk = np.zeros(16, dtype=np.uint8)
    out = np.zeros((1, 16, 8, L1), dtype=np.uint64)
    assert ctx.L.tac_aes_decrypt_public_blocks(ctx.h, 1, 2, blk.ctypes.data, None, out.ctypes.data) == TAC_ERR_STATE
    assert ctx.L.tac_aes_decrypt_blocks(ctx.h, 1, 2, 1, out.ctypes.data, out.ctypes.data) == TAC_ERR_STATE
    assert "tac_aes_inv_key_schedule" in ctx.last_error()


@pytest.mark.gpu
def test_stale_after_set_key_schedule(gpu64, ol):
    ck, ctx = gpu64
    ctx.aes_set_key_schedule(clear_key_schedule_cts(ck, ol, CLI_KEY))
    ctx.aes_inv_key_schedule()
    ctx.aes_decrypt_public_blocks(seeded_blocks(1), rounds=1)
    ctx.aes_set_key_schedule(clear_key_schedule_cts(ck, ol, CLI_KEY))
    with pytest.raises(RuntimeError, match="tac_aes_inv_key_schedule"):
        ctx.aes_decrypt_public_blocks(seeded_blocks(1), rounds=1)
