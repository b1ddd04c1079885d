"""AES over public blocks (AES-CTR keystream and transciphering): the sharing plan against a brute-force restatement of its
rule on the CPU, and on the B200 the device path against clear AES and, word for word, against the encrypted-block path
fed trivial ciphertexts of the same blocks."""
import numpy as np
import pytest

from test_oracle_golden import CLI_IV, CLI_KEY, CLI_OUT

TAC_ERR_ARG = -2


# ---------------------------------------------------------------------------------------------- the plan (host only)
def dependence_sets(rounds):
    """D(r, j) for r = 1..rounds: D(1, j) = {j}, D(r+1, (row, c)) = U_{r'} D(r, 4((c + r') mod 4) + r')"""
    D = [{j} for j in range(16)]
    out = [D]
    for _ in range(1, rounds):
        D = [set().union(*(D[4 * (((j >> 2) + rr) & 3) + rr] for rr in range(4))) for j in range(16)]
        out.append(D)
    return out


def brute_force_plan(blocks, rounds=10):
    blocks = [bytes(b) for b in blocks]
    return [sum(len({tuple(b[i] for i in sorted(D[j])) for b in blocks}) for j in range(16)) for D in dependence_sets(rounds)]


def counters(first, n):
    return [CLI_IV + (first + i).to_bytes(8, "big") for i in range(n)]


def test_dependence_sets_cover_everything_from_round_3():
    D = dependence_sets(3)
    assert D[1][0] == {0, 5, 10, 15} and D[1][7] == {3, 4, 9, 14}
    assert all(d == set(range(16)) for d in D[2])


@pytest.mark.parametrize("first,n,want3", [(1, 128, [143, 524, 2048]), (1, 10, [25, 52, 160]), (200, 128, [144, 528, 2048])])
def test_plan_counter_blocks(tac, first, n, want3):
    blocks = counters(first, n)
    got = tac.aes_public_plan(blocks)
    assert got == brute_force_plan(blocks) == want3 + [16 * n] * 7
    assert got[3:] == [16 * n] * 7


def test_plan_identical_blocks(tac):
    blocks = [CLI_IV * 2] * 5
    assert tac.aes_public_plan(blocks) == brute_force_plan(blocks) == [16] * 10


def test_plan_random_blocks(tac):
    blocks = [np.random.default_rng(3).bytes(16 * 64)[16 * i:16 * i + 16] for i in range(64)]
    got = tac.aes_public_plan(blocks)
    assert got == brute_force_plan(blocks)
    assert got[1:] == [16 * 64] * 9


def test_plan_mixed_and_reduced_rounds(tac):
    blocks = counters(1, 20) + counters(1, 3) + [bytes(16), bytes(16)]     # duplicates, and a block sharing nothing
    for rounds in (1, 2, 10):
        assert tac.aes_public_plan(blocks, rounds) == brute_force_plan(blocks, rounds)
    assert tac.aes_public_plan(counters(1, 128), 1) == [143]
    assert tac.aes_public_plan(counters(1, 128), 2) == [143, 524]
    assert tac.aes_public_plan([], 10) == [0] * 10


def test_plan_argument_errors(tac):
    for rounds in (0, 11):
        with pytest.raises(ValueError):
            tac.aes_public_plan(counters(1, 2), rounds)
    L = tac.load_library()
    boxes = np.zeros(10, dtype=np.int64)
    blk = np.zeros(16, dtype=np.uint8)
    assert L.tac_aes_public_plan(-1, 10, blk.ctypes.data, boxes.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_public_plan(1, 10, None, boxes.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_public_plan(0, 10, None, boxes.ctypes.data) == 0
    with pytest.raises(ValueError):
        tac.aes_public_plan(b"\x00" * 17)


def test_ctr_blocks_layout(tac):
    got = tac.ctr_blocks(CLI_IV, 1, 10)
    assert got.shape == (10, 16) and got.dtype == np.uint8
    assert [bytes(r) for r in got] == counters(1, 10)
    top = tac.ctr_blocks(CLI_IV, 2**64 - 2, 2)
    assert bytes(top[1]) == CLI_IV + b"\xff" * 8
    with pytest.raises(ValueError):
        tac.ctr_blocks(CLI_IV, 2**64 - 2, 3)              # the counter would wrap
    with pytest.raises(ValueError):
        tac.ctr_blocks(CLI_IV[:7], 1, 1)
    assert tac.ctr_blocks(CLI_IV, 5, 0).shape == (0, 16)


# ---------------------------------------------------------------------------------------------- the device path
def clear_key_schedule_cts(ck, ol, key):
    return ck.encrypt_bytes(bytes(ol.plain_key_schedule(key)), first_index=1 << 40)


def trivial_blocks(blocks, L1):
    """trivial encryptions (mask 0, body encode_bit) of public blocks: [n][16][8][L1]"""
    b = np.unpackbits(np.frombuffer(b"".join(blocks), dtype=np.uint8).reshape(-1, 16), axis=1).reshape(-1, 16, 8)
    out = np.zeros(b.shape + (L1,), dtype=np.uint64)
    out[..., -1] = b.astype(np.uint64) << np.uint64(63)
    return out


@pytest.mark.gpu
def test_cli_counters_clear_key_schedule(gpu64, ol):
    ck, ctx = gpu64
    ctx.aes_set_key_schedule(clear_key_schedule_cts(ck, ol, CLI_KEY))
    enc = ctx.aes_ctr_keystream(CLI_IV, 1, 10)
    assert [ck.decrypt_bytes(e).hex() for e in enc] == CLI_OUT


@pytest.mark.gpu
def test_cli_counters_fhe_key_schedule(gpu64, ol):
    ck, ctx = gpu64
    ks = ctx.aes_key_schedule(ck.encrypt_bytes(CLI_KEY, first_index=1 << 42))
    assert ck.decrypt_bytes(ks.reshape(-1, ck.params.big_lwe_size)) == bytes(ol.plain_key_schedule(CLI_KEY))
    enc = ctx.aes_encrypt_public_blocks(counters(1, 10))
    assert [ck.decrypt_bytes(e).hex() for e in enc] == CLI_OUT


def assert_bit_identical(ctx, blocks, rounds):
    L1 = ctx.params.big_lwe_size
    pub = ctx.aes_encrypt_public_blocks(blocks, rounds=rounds)
    ref = ctx.aes_encrypt_blocks(trivial_blocks(blocks, L1), rounds=rounds, in_noise_sq=0)
    assert pub.shape == ref.shape
    bad = np.flatnonzero((pub != ref).any(axis=-1))
    assert bad.size == 0, f"rounds={rounds}: {bad.size} output bits differ, first at {bad[:8].tolist()}"
    return pub


@pytest.mark.gpu
@pytest.mark.parametrize("rounds", [1, 2, 10])
def test_bit_identical_to_encrypted_path(gpu64, tac, ol, rounds):
    """a set that shares in rounds 1 and 2 and holds a duplicate block (shares in every round)"""
    ck, ctx = gpu64
    ctx.aes_set_key_schedule(clear_key_schedule_cts(ck, ol, CLI_KEY))
    blocks = counters(1, 6) + counters(3, 1) + [bytes(range(16))]
    assert all(n < 16 * len(blocks) for n in tac.aes_public_plan(blocks, rounds))
    pub = assert_bit_identical(ctx, blocks, rounds)
    assert np.array_equal(pub[2], pub[6])                        # identical public blocks: word-identical outputs
    for i, b in enumerate(blocks):
        assert ck.decrypt_bytes(pub[i]) == ol.plain_encrypt_block(CLI_KEY, b, rounds)


@pytest.mark.gpu
def test_bit_identical_130_blocks(gpu64, ol):
    """rounds 3+ bootstrap 16·130 = 2080 boxes, more than one pass of the pipeline (2048 boxes at the default max_cts)"""
    ck, ctx = gpu64
    ctx.aes_set_key_schedule(clear_key_schedule_cts(ck, ol, CLI_KEY))
    blocks = counters(200, 130)
    pub = assert_bit_identical(ctx, blocks, 10)
    for i in (0, 57, 129):
        assert ck.decrypt_bytes(pub[i]) == ol.plain_encrypt_block(CLI_KEY, blocks[i])


@pytest.mark.gpu
def test_transcipher_aes_ctr_message(gpu64, ol):
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    ck, ctx = gpu64
    ctx.aes_set_key_schedule(clear_key_schedule_cts(ck, ol, CLI_KEY))
    msg = b"transciphering: AES-CTR in, FHE out."
    msg += b"!" * (37 - len(msg))
    first_ctr = 2**64 - 3                                        # the three blocks end on the last counter
    nonce = CLI_IV + first_ctr.to_bytes(8, "big")
    ct = Cipher(algorithms.AES(CLI_KEY), modes.CTR(nonce)).encryptor().update(msg)
    out = ctx.aes_ctr_transcipher(CLI_IV, first_ctr, ct)
    assert out.shape == (37, 8, ck.params.big_lwe_size)
    assert ck.decrypt_bytes(out) == msg


@pytest.mark.gpu
def test_device_entry_point_and_errors(gpu64, ol):
    import torch
    ck, ctx = gpu64
    ctx.aes_set_key_schedule(clear_key_schedule_cts(ck, ol, CLI_KEY))
    blocks = counters(1, 3)
    out = torch.empty((3, 16, 8, ck.params.big_lwe_size), dtype=torch.int64, device="cuda:0")
    ctx.aes_encrypt_public_blocks_dev(blocks, out.data_ptr(), rounds=2)
    ctx.sync()
    host = ctx.aes_encrypt_public_blocks(blocks, rounds=2)
    assert np.array_equal(out.cpu().numpy().view(np.uint64), host)
    L = ctx.L
    blk = np.zeros(16, dtype=np.uint8)
    for n, rounds, ptr in ((-1, 10, blk.ctypes.data), (1, 0, blk.ctypes.data), (1, 11, blk.ctypes.data), (1, 10, None)):
        assert L.tac_aes_encrypt_public_blocks(ctx.h, n, rounds, ptr, None, host.ctypes.data) == TAC_ERR_ARG


@pytest.mark.gpu
def test_public_path_noise_guard(tac):
    """params_sqrd_lvl_4 cannot hold the S-box outputs' squared noise 9: NoiseTooBig, as on the encrypted-block path"""
    ck = tac.ClientKey(4, seed=1).gen_eval_keys()
    ctx = tac.FheContext(ck.params)
    ctx.upload_keys(ck)
    ctx.aes_set_key_schedule(np.zeros((44, 4, 8, ck.params.big_lwe_size), dtype=np.uint64))
    with pytest.raises(tac.NoiseTooBig):
        ctx.aes_encrypt_public_blocks(counters(1, 1), rounds=2)
