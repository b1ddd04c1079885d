"""AES-GCM transciphering with the tag checked under FHE (NIST SP 800-38D, AES-128, 96-bit IVs).

CPU: the formatting (tac_aes_gcm_format) replayed in clear AES plus a clear GHASH gives the ciphertext and tag of
`cryptography`'s AESGCM for payload and AAD lengths 0..100 and tags of 4, 8, 12 and 16 bytes; Test Cases 1-4 of the GCM
specification; every argument error before any device call.  B200: the encrypted GF(2^128) product against the clear one,
with the largest phase error of its output bits; the GHASH key table of two keys; one batched call over the published
vectors, edge shapes, records longer than the table depth and four tampered records; records under three interleaved keys
against their single-key runs; and the state errors of a missing or stale table."""
import numpy as np
import pytest

from conftest import SEED
from test_aes_ccm import ecb, flip, signed, xor
from test_aes_multikey import RANDOM_KEY, assert_words_equal, schedule_cts

TAC_ERR_ARG, TAC_ERR_STATE = -2, -3

TC_KEY = bytes.fromhex("feffe9928665731c6d6a8f9467308308")
TC_IV = bytes.fromhex("cafebabefacedbaddecaf888")
TC_P = bytes.fromhex("d9313225f88406e5a55909c5aff5269a86a7a9531534f7da2e4c303d8a318a72"
                     "1c3c0c95956809532fcf0e2449a6b525b16aedf5aa0de657ba637b391aafd255")
TC_C = bytes.fromhex("42831ec2217774244b7221b784d0d49ce3aa212f2c02a4e035c17e2329aca12e"
                     "21d514b25466931c7d8f6a5aac84aa051ba30b396a0aac973d58e091473f5985")
# Test Cases 1-4 of "The Galois/Counter Mode of Operation (GCM)" (McGrew, Viega): (key, iv, aad, plaintext, C ‖ T)
VECTORS = {
    "tc1": (bytes(16), bytes(12), b"", b"", bytes.fromhex("58e2fccefa7e3061367f1d57a4e7455a")),
    "tc2": (bytes(16), bytes(12), b"", bytes(16), bytes.fromhex("0388dace60b6a392f328c2b971b2fe78ab6e47d42cec13bdf53a67b21257bddf")),
    "tc3": (TC_KEY, TC_IV, b"", TC_P, TC_C + bytes.fromhex("4d5c2af327cd64a62cf35abd2ba6fab4")),
    "tc4": (TC_KEY, TC_IV, bytes.fromhex("feedfacedeadbeeffeedfacedeadbeefabaddad2"), TC_P[:60],
            TC_C[:60] + bytes.fromhex("5bc94fbc3221a5db94fae95ae7121a47")),
}
DEPTH = 8


def aesgcm(key, iv, pt, tag_len, aad):
    from cryptography.hazmat.primitives.ciphers.aead import AESGCM
    out = AESGCM(key).encrypt(iv, pt, aad or None)
    return out[:len(pt) + tag_len]


def gmul(x, y):
    """GF(2^128) product of two blocks as big-endian integers (SP 800-38D §6.3)"""
    z, v = 0, y
    for i in range(127, -1, -1):
        if (x >> i) & 1:
            z ^= v
        v = (v >> 1) ^ (0xE1 << 120) if v & 1 else v >> 1
    return z


def ghash(h, blocks):
    y = 0
    for b in blocks:
        y = gmul(y ^ int.from_bytes(bytes(b), "big"), h)
    return y


def replay(tac, key, iv, pt, tag_len, aad):
    """AES-GCM encryption in clear AES from tac_aes_gcm_format's blocks"""
    E = ecb(key)
    ctr, _ = tac.aes_gcm_format(iv, bytes(len(pt) + tag_len), tag_len, aad)
    assert ctr.shape == ((len(pt) + 15) // 16 + 1, 16)
    c = xor(pt, b"".join(E(b) for b in ctr[1:]))
    _, blocks = tac.aes_gcm_format(iv, c + bytes(tag_len), tag_len, aad)
    s = ghash(int.from_bytes(E(bytes(16)), "big"), blocks)
    return c + xor(E(ctr[0]), s.to_bytes(16, "big"))[:tag_len]


# ---------------------------------------------------------------------------------------------- formatting (host only)
@pytest.mark.parametrize("name", sorted(VECTORS))
def test_published_vectors(tac, name):
    key, iv, aad, pt, want = VECTORS[name]
    assert aesgcm(key, iv, pt, 16, aad) == want
    assert replay(tac, key, iv, pt, 16, aad) == want


def test_format_replays_aesgcm(tac):
    """payload lengths 0..100 and AAD lengths 0..100, each with the other length and the tag length rotating"""
    rng = np.random.default_rng(SEED)
    key = rng.bytes(16)
    tags = (4, 8, 12, 16)
    cases = [(p, (7 * p) % 101, tags[p % 4]) for p in range(101)] + [((3 * a) % 101, a, tags[a % 4]) for a in range(101)]
    for p, a, t in cases:
        iv, aad, pt = rng.bytes(12), rng.bytes(a), rng.bytes(p)
        assert replay(tac, key, iv, pt, t, aad) == aesgcm(key, iv, pt, t, aad), (p, a, t)


def test_format_blocks(tac):
    iv = bytes(range(1, 13))
    ctr, blocks = tac.aes_gcm_format(iv, bytes(20) + bytes(16), 16, bytes([0xA5]) * 17)
    assert [bytes(c) for c in ctr] == [iv + i.to_bytes(4, "big") for i in (1, 2, 3)]
    assert blocks.shape == (2 + 2 + 1, 16)
    assert bytes(blocks[0]) == bytes([0xA5]) * 16 and bytes(blocks[1]) == b"\xa5" + bytes(15)
    assert bytes(blocks[-1]) == (17 * 8).to_bytes(8, "big") + (20 * 8).to_bytes(8, "big")


def test_argument_errors(tac):
    L = tac.load_library()
    counts = np.zeros(2, dtype=np.int64)

    def fmt(iv_len=12, tag_len=16, aad_len=0, data_len=32, aad=True, data=True, iv=True):
        buf = bytes(max(16, data_len, aad_len))
        ptr = tac.C.cast(tac.C.c_char_p(buf), tac.C.c_void_p).value
        m = tac.CcmMsg(ptr if iv else None, iv_len, tag_len, ptr if aad else None, aad_len, ptr if data else None, data_len)
        return L.tac_aes_gcm_format(tac.C.addressof(m), None, None, counts.ctypes.data)

    assert fmt() == 0 and counts.tolist() == [2, 2]
    for t in (4, 8, 12, 13, 14, 15, 16):
        assert fmt(tag_len=t) == 0, t
    for bad in (dict(iv_len=8), dict(iv_len=16), dict(tag_len=6), dict(tag_len=10), dict(tag_len=2), dict(tag_len=18),
                dict(data_len=7, tag_len=8), dict(iv=False), dict(aad=False, aad_len=1), dict(data=False)):
        assert fmt(**bad) == TAC_ERR_ARG, bad
    # the length limits are checked from the lengths alone (nothing is read for the query)
    big = tac.CcmMsg(tac.C.cast(tac.C.c_char_p(bytes(16)), tac.C.c_void_p).value, 12, 16, None, 0,
                     tac.C.cast(tac.C.c_char_p(bytes(16)), tac.C.c_void_p).value, (1 << 36) - 32 + 16 + 1)
    assert L.tac_aes_gcm_format(tac.C.addressof(big), None, None, counts.ctypes.data) == TAC_ERR_ARG
    big_aad = tac.CcmMsg(big.nonce, 12, 16, big.nonce, 1 << 61, big.data, 16)
    assert L.tac_aes_gcm_format(tac.C.addressof(big_aad), None, None, counts.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_gcm_format(None, None, None, counts.ctypes.data) == TAC_ERR_ARG
    bad_records = [(bytes(8), bytes(20), 16, b""), (bytes(16), bytes(20), 16, b""), (bytes(12), bytes(20), 6, b""),
                   (bytes(12), bytes(20), 18, b""), (bytes(12), bytes(7), 8, b""), (bytes(12), bytes(20), 16.0, b"")]
    for iv, data, t, aad in bad_records:
        with pytest.raises(ValueError):
            tac.aes_gcm_format(iv, data, t, aad)
    # the context's checks run before any device call: this object has no device state at all
    ctx = object.__new__(tac.FheContext)
    ctx.L, ctx.params = L, tac.params_preset(64)
    ctx._n_keys = 2
    for iv, data, t, aad in bad_records:
        with pytest.raises(ValueError):
            ctx.aes_gcm_transcipher(iv, data, t, aad)
        with pytest.raises(ValueError):
            ctx.aes_gcm_transcipher_many([(0, bytes(12), bytes(20), 16, b""), (1, iv, data, t, aad)])
    for k in (-1, 2, 0.5):
        with pytest.raises(ValueError):
            ctx.aes_gcm_transcipher_many([(0, bytes(12), bytes(20), 16, b""), (k, bytes(12), bytes(20), 16, b"")])
    for depth in (0, 3, 6, 2048, 8.0):
        with pytest.raises(ValueError):
            ctx.aes_gcm_hash_key(depth)
        with pytest.raises(ValueError):
            ctx.aes_gcm_hash_key_table(depth)


# ---------------------------------------------------------------------------------------------- the device path
@pytest.fixture(scope="module")
def client(tac):
    """a second client on the session's lvl-64 secret keys (same seed) for this file's encryptions: the session client's
    encryption counter, which later tests' default-indexed encryptions follow, stays as it was"""
    return tac.ClientKey(64, seed=SEED)


def block_int(ck, bits):
    return int.from_bytes(ck.decrypt_bytes(np.asarray(bits).reshape(16, 8, -1)), "big")


def phase_error(ck, cts, bits):
    want = np.asarray(bits, dtype=np.uint64) << np.uint64(63)
    return float(np.abs(signed(ck.decrypt_phases(cts.reshape(-1, cts.shape[-1])) - want)).max())


@pytest.mark.gpu
def test_gf128_mul(tac, gpu64, client):
    ck, ctx = client, gpu64[1]
    rng = np.random.default_rng(SEED + 10)
    vals = [rng.bytes(16) for _ in range(5)]
    one, x127, zero = (1 << 127).to_bytes(16, "big"), (1).to_bytes(16, "big"), bytes(16)
    pairs = [(vals[0], vals[1]), (vals[2], vals[3]), (vals[4], zero), (vals[0], one), (one, vals[1]), (x127, x127), (x127, vals[2])]
    a = np.stack([ck.encrypt_bytes(p, first_index=(1 << 54) + 256 * i) for i, (p, _) in enumerate(pairs)]).reshape(len(pairs), 128, -1)
    b = np.stack([ck.encrypt_bytes(q, first_index=(1 << 54) + 256 * i + 128) for i, (_, q) in enumerate(pairs)]).reshape(len(pairs), 128, -1)
    out = ctx.gf128_mul(a, b)
    worst = 0.0
    for i, (p, q) in enumerate(pairs):
        want = gmul(int.from_bytes(p, "big"), int.from_bytes(q, "big"))
        assert block_int(ck, out[i]) == want, i
        bits = [(want >> (127 - j)) & 1 for j in range(128)]
        worst = max(worst, phase_error(ck, out[i], bits))
    print(f"GF(2^128) product: largest output phase error 2^{np.log2(worst + 1):.1f}")
    assert worst < 2.0 ** 59


@pytest.mark.gpu
def test_hash_key_table_powers(tac, gpu64, client, ol):
    ck, ctx = client, gpu64[1]
    keys = [TC_KEY, RANDOM_KEY]
    ctx.aes_set_key_table(schedule_cts(ck, ol, keys, 1 << 55))
    table = ctx.aes_gcm_hash_key_table(DEPTH)
    assert table.shape == (2, DEPTH, 128, ck.params.big_lwe_size)
    for k, key in enumerate(keys):
        h = int.from_bytes(ecb(key)(bytes(16)), "big")
        p = h
        for e in range(1, DEPTH + 1):
            assert block_int(ck, table[k, e - 1]) == p, (k, e)
            p = gmul(p, h)


def record(key, iv, pt, t, aad):
    return dict(key=key, iv=iv, aad=aad, t=t, data=aesgcm(key, iv, pt, t, aad), pt=pt, genuine=True)


def batch_records():
    """the published vectors, edge shapes, records longer than the table depth and four tampered records, two keys"""
    rng = np.random.default_rng(SEED + 11)
    recs = [record(*VECTORS[n][:2], VECTORS[n][3], 16, VECTORS[n][2]) for n in sorted(VECTORS)]
    recs.append(record(TC_KEY, rng.bytes(12), b"", 16, rng.bytes(20)))                       # GMAC: no payload
    recs.append(record(RANDOM_KEY, rng.bytes(12), rng.bytes(37), 12, b""))                  # no AAD
    recs.append(record(TC_KEY, rng.bytes(12), rng.bytes(150), 16, rng.bytes(13)))           # M = 12 > depth: one product
    recs.append(record(RANDOM_KEY, rng.bytes(12), rng.bytes(260), 4, rng.bytes(3)))        # M = 19: two products
    base = record(TC_KEY, rng.bytes(12), rng.bytes(64), 16, rng.bytes(13))
    ct_flip = dict(base, data=flip(base["data"], 21), pt=flip(base["pt"], 21), genuine=False)
    tag = record(RANDOM_KEY, rng.bytes(12), rng.bytes(20), 8, rng.bytes(5))
    tag_flip = dict(tag, data=flip(tag["data"], 8 * 20 + 3), genuine=False)
    aad = record(TC_KEY, rng.bytes(12), rng.bytes(16), 16, rng.bytes(30))
    aad_alt = dict(aad, aad=flip(aad["aad"], 9), genuine=False)
    iv = record(RANDOM_KEY, rng.bytes(12), rng.bytes(33), 13, rng.bytes(3))
    iv_alt = dict(iv, iv=flip(iv["iv"], 0), genuine=False)
    return recs + [ct_flip, tag_flip, aad_alt, iv_alt]


def ctr_plaintext(tac, key, iv, data, t):
    ctr, _ = tac.aes_gcm_format(iv, data, t)
    E = ecb(key)
    return xor(data[:len(data) - t], b"".join(E(c) for c in ctr[1:]))


@pytest.mark.gpu
def test_batched_records_and_tampering(tac, gpu64, client, ol):
    ck, ctx = client, gpu64[1]
    L1 = ck.params.big_lwe_size
    keys = [bytes(16), TC_KEY, RANDOM_KEY]
    scheds = schedule_cts(ck, ol, keys, 1 << 56)
    ctx.aes_set_key_table(scheds)
    ctx.aes_gcm_hash_key_table(DEPTH)
    recs = batch_records()
    msgs = [(keys.index(r["key"]), r["iv"], r["data"], r["t"], r["aad"]) for r in recs]
    out = ctx.aes_gcm_transcipher_many(msgs)
    assert len(out) == len(recs)
    worst = 0.0
    for i, (r, (pt, valid)) in enumerate(zip(recs, out)):
        p = len(r["data"]) - r["t"]
        assert pt.shape == (p, 8, L1) and valid.shape == (L1,), i
        want_pt = ctr_plaintext(tac, r["key"], r["iv"], r["data"], r["t"])
        if i != len(recs) - 1:
            assert want_pt == r["pt"], i
        assert ck.decrypt_bytes(pt) == want_pt, i
        bit = int(ck.decrypt_bits(valid)[0])
        assert bit == int(r["genuine"]), (i, bit)
        worst = max(worst, phase_error(ck, valid[None], [bit]))
        if p:
            ctr, _ = tac.aes_gcm_format(r["iv"], r["data"], r["t"], r["aad"])
            m = ctr.shape[0] - 1
            ref = ctx.aes_encrypt_public_blocks_keyed(ctr[1:], [msgs[i][0]] * m, xor=r["data"][:p] + bytes(16 * m - p))
            assert_words_equal(pt, ref.reshape(-1, 8, L1)[:p], f"record {i} against aes_encrypt_public_blocks_keyed")
    print(f"largest validity-bit phase error: 2^{np.log2(worst + 1):.1f}")
    assert worst < 2.0 ** 59
    for i in (1, 6, 7, len(recs) - 3):
        (pt, valid), = ctx.aes_gcm_transcipher_many([msgs[i]])
        assert_words_equal(pt, out[i][0], f"record {i} alone, plaintext")
        assert_words_equal(valid[None], out[i][1][None], f"record {i} alone, validity bit")
    ctx.aes_set_key_schedule(scheds[1])
    ctx.aes_gcm_hash_key(DEPTH)
    r = recs[3]
    assert r["key"] == TC_KEY
    pt, valid = ctx.aes_gcm_transcipher(r["iv"], r["data"], r["t"], r["aad"])
    assert_words_equal(pt, out[3][0], "Test Case 4 under the single schedule, plaintext")
    assert_words_equal(valid[None], out[3][1][None], "Test Case 4 under the single schedule, validity bit")


@pytest.mark.gpu
def test_records_under_three_keys(tac, gpu64, client, ol):
    """chunk counts 1..3 interleaved over three table entries: every record gets the words of its own single-key run"""
    ck, ctx = client, gpu64[1]
    keys = [TC_KEY, bytes(16), RANDOM_KEY]
    scheds = schedule_cts(ck, ol, keys, 1 << 57)
    ctx.aes_set_key_table(scheds)
    ctx.aes_gcm_hash_key_table(DEPTH)
    rng = np.random.default_rng(SEED + 12)
    shapes = [(2, 13, 64), (0, 0, 200), (1, 5, 16), (2, 40, 100), (0, 13, 0), (1, 0, 130)]    # key, |A|, p
    recs = []
    for i, (k, a, p) in enumerate(shapes):
        r = record(keys[k], rng.bytes(12), rng.bytes(p), 16, rng.bytes(a))
        recs.append(dict(r, data=flip(r["data"], 8 * p + 1)) if i == 3 else r)
    out = ctx.aes_gcm_transcipher_many([(k, r["iv"], r["data"], 16, r["aad"]) for (k, _, _), r in zip(shapes, recs)])
    for k in range(3):
        ctx.aes_set_key_schedule(scheds[k])
        ctx.aes_gcm_hash_key(DEPTH)
        for i, ((kk, _, _), r, (pt, valid)) in enumerate(zip(shapes, recs, out)):
            if kk != k:
                continue
            assert ck.decrypt_bytes(pt) == r["pt"], i
            assert int(ck.decrypt_bits(valid)[0]) == (i != 3), i
            spt, svalid = ctx.aes_gcm_transcipher(r["iv"], r["data"], 16, r["aad"])
            assert_words_equal(pt, spt, f"record {i}: plaintext against its single-key run")
            assert_words_equal(valid[None], svalid[None], f"record {i}: validity bit against its single-key run")


@pytest.mark.gpu
def test_state_errors(tac, ck64, client, ol):
    ctx = tac.FheContext(ck64.params, device=0)
    L = ctx.L
    msgs, keep, _ = tac._gcm_messages([(bytes(12), bytes(32), 16, b"")])
    L1 = ck64.params.big_lwe_size
    pt, valid = np.zeros((16, 8, L1), dtype=np.uint64), np.zeros(L1, dtype=np.uint64)
    kidx = np.zeros(1, dtype=np.int32)
    assert L.tac_aes_gcm_transcipher(ctx.h, 1, None, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_STATE
    assert L.tac_aes_gcm_hash_key(ctx.h, 8, None) == TAC_ERR_STATE                       # no keys
    ctx.upload_keys(ck64)
    assert L.tac_aes_gcm_hash_key(ctx.h, 8, None) == TAC_ERR_STATE                       # no schedule
    assert L.tac_aes_gcm_hash_key_table(ctx.h, 8, None) == TAC_ERR_STATE                 # no key table
    sched = schedule_cts(client, ol, [RANDOM_KEY], 1 << 58)
    ctx.aes_set_key_schedule(sched[0])
    ctx.aes_set_key_table(sched)
    assert L.tac_aes_gcm_hash_key(ctx.h, 6, None) == TAC_ERR_ARG
    assert L.tac_aes_gcm_transcipher(ctx.h, 1, None, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_STATE          # no table
    assert L.tac_aes_gcm_transcipher(ctx.h, 1, kidx.ctypes.data, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_STATE
    ctx.aes_gcm_hash_key(1)
    ctx.aes_gcm_hash_key_table(1)
    pt1, v1 = ctx.aes_gcm_transcipher(bytes(12), bytes(32))
    ctx.aes_set_key_schedule(sched[0])                                                  # the single table is stale now
    assert L.tac_aes_gcm_transcipher(ctx.h, 1, None, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_STATE
    assert L.tac_aes_gcm_transcipher(ctx.h, 1, kidx.ctypes.data, msgs, pt.ctypes.data, valid.ctypes.data) == 0
    ctx.aes_set_key_table(sched)                                                        # and now the keyed one
    launches = ctx.launch_count()
    assert L.tac_aes_gcm_transcipher(ctx.h, 1, kidx.ctypes.data, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_STATE
    assert ctx.launch_count() == launches
    small = tac.FheContext(4, device=0)
    with pytest.raises(tac.NoiseTooBig):
        small.aes_gcm_transcipher(bytes(12), bytes(32))
