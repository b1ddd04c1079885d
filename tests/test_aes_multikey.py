"""AES under many keys: a resident table of key schedules, batched key expansion, and keyed calls in which every block
names its key.

CPU: the keyed sharing plan against a brute-force restatement of its rule (a group is the key and the bytes of D(r, j)),
its reduction to the single-key plan, and the argument checks that run before any device call.  B200: the batched key
expansion against clear schedules and against the single-key expansion, keyed encryption / decryption / transciphering
against clear AES and, word for word, against the single-key paths, and the state rules of the table."""
import numpy as np
import pytest

from test_aes_decrypt import FIPS_CT, FIPS_KEY, FIPS_PT, clear_inv_key_schedule, dependence_sets, plain_decrypt_block, seeded_blocks
from conftest import SEED
from test_oracle_golden import CLI_IV, CLI_KEY

TAC_ERR_ARG, TAC_ERR_STATE = -2, -3

RANDOM_KEY = bytes.fromhex("8e73b0f7da0e6452c810f32b809079e5")


# ---------------------------------------------------------------------------------------------- the keyed plan (host only)
def brute_force_keyed_plan(blocks, key_index, rounds=10, inverse=False):
    blocks = [bytes(b) for b in blocks]
    return [sum(len({(k, tuple(b[i] for i in sorted(D[j]))) for b, k in zip(blocks, key_index)}) for j in range(16))
            for D in dependence_sets(rounds, inverse)]


def counters(first, n, iv=CLI_IV):
    return [iv + (first + i).to_bytes(8, "big") for i in range(n)]


@pytest.mark.parametrize("inverse", [False, True])
def test_keyed_plan_brute_force(tac, inverse):
    rng = np.random.default_rng(17)
    distinct = seeded_blocks(12, seed=41)
    blocks = distinct + distinct[:6] + counters(1, 20)                          # repeats under the same or another key
    key_index = [int(k) for k in rng.integers(0, 3, size=len(blocks))]
    for rounds in (1, 2, 10):
        got = tac.aes_public_plan(blocks, rounds, decrypt=inverse, key_index=key_index)
        assert got == brute_force_keyed_plan(blocks, key_index, rounds, inverse)


def test_keyed_plan_without_keys_is_the_plan(tac):
    L = tac.load_library()
    blocks = counters(1, 128) + seeded_blocks(5, seed=2) + [bytes(16)] * 3
    b = np.frombuffer(b"".join(blocks), dtype=np.uint8).copy()
    zeros = np.zeros(len(blocks), dtype=np.int32)
    for decrypt in (0, 1):
        want = np.zeros(10, dtype=np.int64)
        (L.tac_aes_public_plan_inv if decrypt else L.tac_aes_public_plan)(len(blocks), 10, b.ctypes.data, want.ctypes.data)
        for kidx in (None, zeros.ctypes.data):
            got = np.zeros(10, dtype=np.int64)
            assert L.tac_aes_public_plan_keyed(len(blocks), 10, decrypt, kidx, b.ctypes.data, got.ctypes.data) == 0
            assert np.array_equal(got, want)
        assert tac.aes_public_plan(blocks, decrypt=bool(decrypt), key_index=[0] * len(blocks)) == [int(v) for v in want]


def test_identical_counters_under_two_keys_share_nothing(tac):
    one = tac.aes_public_plan(counters(1, 64))
    both = tac.aes_public_plan(counters(1, 64) * 2, key_index=[0] * 64 + [1] * 64)
    assert both == [2 * n for n in one]
    assert tac.aes_public_plan(counters(1, 64) * 2, key_index=[5] * 128) == tac.aes_public_plan(counters(1, 64))


def test_keyed_argument_errors(tac):
    L = tac.load_library()
    boxes = np.zeros(10, dtype=np.int64)
    blk = np.zeros(32, dtype=np.uint8)
    assert L.tac_aes_public_plan_keyed(2, 10, 0, np.array([0, -1], dtype=np.int32).ctypes.data, blk.ctypes.data, boxes.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_public_plan_keyed(2, 10, 1, np.array([-7, 0], dtype=np.int32).ctypes.data, blk.ctypes.data, boxes.ctypes.data) == TAC_ERR_ARG
    with pytest.raises(ValueError):
        tac.aes_public_plan(counters(1, 2), key_index=[0, -1])
    with pytest.raises(ValueError):
        tac.aes_public_plan(counters(1, 2), key_index=[0])
    # the context's checks run before any device call: this object has no device state at all
    ctx = object.__new__(tac.FheContext)
    ctx.L, ctx.params = L, tac.params_preset(64)
    ctx._n_keys = 2
    for kidx in ([0, -1], [0, 2], None, [0]):
        with pytest.raises(ValueError):
            ctx.aes_encrypt_public_blocks_keyed(counters(1, 2), kidx)
        with pytest.raises(ValueError):
            ctx.aes_decrypt_public_blocks_keyed(counters(1, 2), kidx)
    with pytest.raises(ValueError):
        ctx.aes_ctr_transcipher_many([(2, CLI_IV, 1, b"x")])
    with pytest.raises(ValueError):
        ctx.aes_cbc_transcipher_many([(-1, bytes(16), bytes(16))])
    with pytest.raises(ValueError):
        ctx.aes_cbc_transcipher_many([(0, bytes(16), bytes(17))])
    with pytest.raises(ValueError):
        ctx.aes_set_key_table(np.zeros(0, dtype=np.uint64))                 # n_keys < 1
    with pytest.raises(ValueError):
        ctx.aes_key_table(np.zeros(0, dtype=np.uint64))
    with pytest.raises(ValueError):
        ctx.aes_set_inv_key_table(np.zeros((1, 44, 4, 8, ctx.params.big_lwe_size), dtype=np.uint64))   # 1 schedule for 2 keys


# ---------------------------------------------------------------------------------------------- the device path
KEYS = (FIPS_KEY, CLI_KEY, RANDOM_KEY)


@pytest.fixture(scope="module")
def client(tac):
    """a second client on the session's lvl-64 secret keys (same seed) for this file's encryptions: the session client's
    encryption counter, which later tests' default-indexed encryptions follow, stays as it was"""
    return tac.ClientKey(64, seed=SEED)


def schedule_cts(ck, ol, keys, first):
    """client-encrypted clear key schedules [K][44][4][8][L1]"""
    return np.stack([ck.encrypt_bytes(bytes(ol.plain_key_schedule(k)), first_index=first + i * 2048).reshape(44, 4, 8, -1)
                     for i, k in enumerate(keys)])


def inv_schedule_cts(ck, ol, keys, first):
    return np.stack([ck.encrypt_bytes(clear_inv_key_schedule(ol, k), first_index=first + i * 2048).reshape(44, 4, 8, -1)
                     for i, k in enumerate(keys)])


def with_clear_tables(ck, ctx, ol, keys=KEYS):
    ctx.aes_set_key_table(schedule_cts(ck, ol, keys, 1 << 45))
    ctx.aes_set_inv_key_table(inv_schedule_cts(ck, ol, keys, 1 << 46))


def block_cts(ck, blocks, first=1 << 47):
    return np.stack([ck.encrypt_bytes(b, first_index=first + 128 * i) for i, b in enumerate(blocks)])


def assert_words_equal(a, b, what):
    assert a.shape == b.shape, what
    bad = np.flatnonzero((a != b).any(axis=-1))
    assert bad.size == 0, f"{what}: {bad.size} bit ciphertexts differ, first at {bad[:8].tolist()}"


@pytest.mark.gpu
def test_key_table_of_three_keys(gpu64, client, ol):
    ck, ctx = client, gpu64[1]
    L1 = ck.params.big_lwe_size
    key_bits = np.stack([ck.encrypt_bytes(k, first_index=(1 << 48) + 128 * i) for i, k in enumerate(KEYS)])
    table = ctx.aes_key_table(key_bits)
    assert table.shape == (3, 44, 4, 8, L1) and ctx.n_keys == 3
    for i, k in enumerate(KEYS):
        assert ck.decrypt_bytes(table[i].reshape(-1, L1)) == bytes(ol.plain_key_schedule(k)), i
    single = ctx.aes_key_schedule(key_bits[0])
    assert_words_equal(single, table[0], "entry 0 against tac_aes_key_schedule")
    dk = ctx.aes_inv_key_table()
    for i, k in enumerate(KEYS):
        assert ck.decrypt_bytes(dk[i].reshape(-1, L1)) == clear_inv_key_schedule(ol, k), i
    assert_words_equal(ctx.aes_inv_key_schedule(), dk[0], "inverse entry 0 against tac_aes_inv_key_schedule")


@pytest.mark.gpu
def test_keyed_encryption_of_interleaved_blocks(gpu64, client, ol):
    ck, ctx = client, gpu64[1]
    with_clear_tables(ck, ctx, ol)
    key_index = [2, 0, 1, 0, 2, 1, 0]
    blocks = seeded_blocks(len(key_index), seed=77)
    blocks[1] = FIPS_PT                                                          # under FIPS_KEY: FIPS-197 C.1
    cts = block_cts(ck, blocks)
    out = ctx.aes_encrypt_blocks_keyed(cts, key_index)
    for i, (b, k) in enumerate(zip(blocks, key_index)):
        assert ck.decrypt_bytes(out[i]) == ol.plain_encrypt_block(KEYS[k], b, 10), i
    assert ck.decrypt_bytes(out[1]) == FIPS_CT
    scheds = schedule_cts(ck, ol, KEYS, 1 << 45)
    for k in range(3):
        sel = [i for i, kk in enumerate(key_index) if kk == k]
        ctx.aes_set_key_schedule(scheds[k])
        assert_words_equal(out[sel], ctx.aes_encrypt_blocks(cts[sel]), f"key {k} against the single-key path")


@pytest.mark.gpu
def test_one_key_equals_the_unkeyed_entry_points(gpu64, client, ol):
    import torch
    ck, ctx = client, gpu64[1]
    with_clear_tables(ck, ctx, ol, keys=(CLI_KEY,))
    ctx.aes_set_key_schedule(schedule_cts(ck, ol, (CLI_KEY,), 1 << 45)[0])
    ctx.aes_set_inv_key_schedule(inv_schedule_cts(ck, ol, (CLI_KEY,), 1 << 46)[0])
    blocks = seeded_blocks(3, seed=55)
    zeros = [0, 0, 0]
    cts = block_cts(ck, blocks)
    xor = blocks[::-1]
    for rounds in (2, 10):
        assert_words_equal(ctx.aes_encrypt_blocks_keyed(cts, zeros, rounds), ctx.aes_encrypt_blocks(cts, rounds), "encrypt_blocks")
        assert_words_equal(ctx.aes_decrypt_blocks_keyed(cts, zeros, rounds), ctx.aes_decrypt_blocks(cts, rounds), "decrypt_blocks")
        assert_words_equal(ctx.aes_encrypt_public_blocks_keyed(blocks, zeros, rounds, xor=xor),
                           ctx.aes_encrypt_public_blocks(blocks, rounds, xor=xor), "encrypt_public_blocks")
        assert_words_equal(ctx.aes_decrypt_public_blocks_keyed(blocks, zeros, rounds, xor=xor),
                           ctx.aes_decrypt_public_blocks(blocks, rounds, xor=xor), "decrypt_public_blocks")
    # the _dev forms write the same words into device memory
    L1 = ck.params.big_lwe_size
    out = torch.empty((3, 16, 8, L1), dtype=torch.int64, device="cuda:0")
    ctx.aes_encrypt_public_blocks_keyed_dev(blocks, zeros, out.data_ptr(), rounds=2, xor=xor)
    ctx.sync()
    assert_words_equal(out.cpu().numpy().view(np.uint64), ctx.aes_encrypt_public_blocks(blocks, 2, xor=xor), "encrypt_public_blocks_keyed_dev")
    ctx.aes_decrypt_public_blocks_keyed_dev(blocks, zeros, out.data_ptr(), rounds=2)
    ctx.sync()
    assert_words_equal(out.cpu().numpy().view(np.uint64), ctx.aes_decrypt_public_blocks(blocks, 2), "decrypt_public_blocks_keyed_dev")
    in_dev = torch.from_numpy(cts.view(np.int64)).to("cuda:0")
    ctx.aes_encrypt_blocks_keyed_dev(3, zeros, in_dev.data_ptr(), out.data_ptr(), rounds=2)
    ctx.sync()
    assert_words_equal(out.cpu().numpy().view(np.uint64), ctx.aes_encrypt_blocks(cts, 2), "encrypt_blocks_keyed_dev")
    ctx.aes_decrypt_blocks_keyed_dev(3, zeros, in_dev.data_ptr(), out.data_ptr(), rounds=2)
    ctx.sync()
    assert_words_equal(out.cpu().numpy().view(np.uint64), ctx.aes_decrypt_blocks(cts, 2), "decrypt_blocks_keyed_dev")


def ctr_encrypt(ol, key, iv, first_ctr, data):
    stream = b"".join(ol.plain_encrypt_block(key, blk, 10) for blk in counters(first_ctr, (len(data) + 15) // 16, iv))
    return bytes(a ^ b for a, b in zip(data, stream))


@pytest.mark.gpu
def test_ctr_many_senders_with_the_same_counters(gpu64, client, tac, ol):
    ck, ctx = client, gpu64[1]
    with_clear_tables(ck, ctx, ol, keys=(CLI_KEY, RANDOM_KEY))
    iv = bytes(range(8))
    msgs = [b"first sender, same counters!" + b"." * 4, b"second sender's message, 2 blk"]
    cts = [ctr_encrypt(ol, k, iv, 5, m) for k, m in zip((CLI_KEY, RANDOM_KEY), msgs)]
    blocks = counters(5, 2, iv) * 2
    assert tac.aes_public_plan(blocks, key_index=[0, 0, 1, 1]) == [2 * n for n in tac.aes_public_plan(counters(5, 2, iv))]
    out = ctx.aes_ctr_transcipher_many([(0, iv, 5, cts[0]), (1, iv, 5, cts[1])])
    assert [o.shape[0] for o in out] == [len(m) for m in msgs]
    assert [ck.decrypt_bytes(o) for o in out] == msgs


@pytest.mark.gpu
def test_cbc_many_senders(gpu64, client, ol):
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    ck, ctx = client, gpu64[1]
    keys = (RANDOM_KEY, CLI_KEY)
    rng = np.random.default_rng(99)
    ivs = [rng.bytes(16), rng.bytes(16)]
    msgs = [b"CBC from sender zero, 2 blocks.!", b"sender one sends three blocks of CBC text here!!"]
    assert [len(m) for m in msgs] == [32, 48]                                   # whole blocks: CBC has no padding here
    cts = [Cipher(algorithms.AES(k), modes.CBC(iv)).encryptor().update(m) for k, iv, m in zip(keys, ivs, msgs)]
    messages = [(1, ivs[1], cts[1]), (0, ivs[0], cts[0])]
    # inverse table derived on the device
    ctx.aes_set_key_table(schedule_cts(ck, ol, keys, 1 << 45))
    ctx.aes_inv_key_table()
    derived = ctx.aes_cbc_transcipher_many(messages)
    assert [ck.decrypt_bytes(o) for o in derived] == [msgs[1], msgs[0]]
    # and uploaded
    ctx.aes_set_inv_key_table(inv_schedule_cts(ck, ol, keys, 1 << 46))
    uploaded = ctx.aes_cbc_transcipher_many(messages)
    assert [ck.decrypt_bytes(o) for o in uploaded] == [msgs[1], msgs[0]]


@pytest.mark.gpu
def test_keyed_call_of_more_than_one_pass(gpu64, client, ol):
    """rounds 3+ bootstrap 16·130 = 2080 boxes, more than one pass of the pipeline (2048 boxes at the default max_cts)"""
    ck, ctx = client, gpu64[1]
    with_clear_tables(ck, ctx, ol)
    blocks = seeded_blocks(130, seed=130)
    key_index = [(7 * i) % 3 for i in range(130)]
    enc = ctx.aes_encrypt_public_blocks_keyed(blocks, key_index)
    dec = ctx.aes_decrypt_public_blocks_keyed(blocks, key_index)
    for i in range(130):
        k = KEYS[key_index[i]]
        assert ck.decrypt_bytes(enc[i]) == ol.plain_encrypt_block(k, blocks[i], 10), i
        assert ck.decrypt_bytes(dec[i]) == plain_decrypt_block(ol, k, blocks[i]), i


@pytest.mark.gpu
def test_state_rules(tac, ck64, client, ol):
    ctx = tac.FheContext(ck64.params, device=0)
    ctx.upload_keys(ck64)
    L = ctx.L
    L1 = ck64.params.big_lwe_size
    blk = np.frombuffer(b"".join(counters(1, 2)), dtype=np.uint8).copy()
    kidx = np.zeros(2, dtype=np.int32)
    out = np.zeros((2, 16, 8, L1), dtype=np.uint64)
    # no key table yet
    assert L.tac_aes_encrypt_public_blocks_keyed(ctx.h, 2, 1, kidx.ctypes.data, blk.ctypes.data, None, out.ctypes.data) == TAC_ERR_STATE
    assert L.tac_aes_inv_key_table(ctx.h, None) == TAC_ERR_STATE
    assert L.tac_aes_set_inv_key_table(ctx.h, out.ctypes.data) == TAC_ERR_STATE
    # the single-key path, then a table beside it
    ctx.aes_set_key_schedule(schedule_cts(client, ol, (CLI_KEY,), 1 << 45)[0])
    ctx.aes_set_inv_key_schedule(inv_schedule_cts(client, ol, (CLI_KEY,), 1 << 46)[0])
    before = ctx.aes_encrypt_public_blocks(counters(1, 2), rounds=1)
    ctx.aes_set_key_table(schedule_cts(client, ol, (RANDOM_KEY, FIPS_KEY), 1 << 49))
    assert_words_equal(ctx.aes_encrypt_public_blocks(counters(1, 2), rounds=1), before, "single-key output after a table call")
    assert client.decrypt_bytes(ctx.aes_decrypt_public_blocks([FIPS_CT])[0]) == plain_decrypt_block(ol, CLI_KEY, FIPS_CT)   # dk still valid
    # decryption needs the inverse table: none yet, then stale after aes_set_key_table
    assert L.tac_aes_decrypt_public_blocks_keyed(ctx.h, 2, 1, kidx.ctypes.data, blk.ctypes.data, None, out.ctypes.data) == TAC_ERR_STATE
    assert "tac_aes_inv_key_table" in ctx.last_error()
    assert L.tac_aes_decrypt_blocks_keyed(ctx.h, 2, 1, 1, kidx.ctypes.data, out.ctypes.data, out.ctypes.data) == TAC_ERR_STATE
    ctx.aes_set_inv_key_table(inv_schedule_cts(client, ol, (RANDOM_KEY, FIPS_KEY), 1 << 50))
    got = ctx.aes_decrypt_public_blocks_keyed([FIPS_CT], [1])
    assert client.decrypt_bytes(got[0]) == FIPS_PT
    ctx.aes_set_key_table(schedule_cts(client, ol, (RANDOM_KEY, FIPS_KEY), 1 << 49))
    assert L.tac_aes_decrypt_public_blocks_keyed(ctx.h, 2, 1, kidx.ctypes.data, blk.ctypes.data, None, out.ctypes.data) == TAC_ERR_STATE
    # a single schedule change leaves the table's inverse table alone, and vice versa
    ctx.aes_inv_key_table()
    ctx.aes_set_key_schedule(schedule_cts(client, ol, (CLI_KEY,), 1 << 45)[0])
    assert client.decrypt_bytes(ctx.aes_decrypt_public_blocks_keyed([FIPS_CT], [1])[0]) == FIPS_PT
    # argument errors fail before anything runs
    launches = ctx.launch_count()
    for bad in ([0, 2], [-1, 0]):
        k = np.array(bad, dtype=np.int32)
        assert L.tac_aes_encrypt_public_blocks_keyed(ctx.h, 2, 10, k.ctypes.data, blk.ctypes.data, None, out.ctypes.data) == TAC_ERR_ARG
        assert L.tac_aes_encrypt_blocks_keyed(ctx.h, 2, 10, 1, k.ctypes.data, out.ctypes.data, out.ctypes.data) == TAC_ERR_ARG
        assert L.tac_aes_decrypt_public_blocks_keyed_dev(ctx.h, 2, 10, k.ctypes.data, blk.ctypes.data, None, None) == TAC_ERR_ARG
    assert "outside [0, 2)" in ctx.last_error()
    assert L.tac_aes_encrypt_public_blocks_keyed(ctx.h, 2, 10, None, blk.ctypes.data, None, out.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_set_key_table(ctx.h, 0, out.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_key_table(ctx.h, 0, out.ctypes.data, None) == TAC_ERR_ARG
    assert L.tac_aes_set_inv_key_table(ctx.h, None) == TAC_ERR_ARG
    assert L.tac_aes_key_schedule(ctx.h, None, None) == TAC_ERR_ARG
    assert ctx.launch_count() == launches
    assert_words_equal(ctx.aes_encrypt_public_blocks(counters(1, 2), rounds=1), before, "single-key output after NULL key bits")
