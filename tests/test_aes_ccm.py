"""AES-CCM transciphering with the tag checked under FHE (NIST SP 800-38C, RFC 3610).

CPU: the formatting (tac_aes_ccm_format) replayed in clear AES, with the real plaintext in the payload blocks, gives the
ciphertext and tag of `cryptography`'s AESCCM for every nonce length, tag length and AAD length class; the published
vectors; and the argument checks that run before any device call.  B200: one batched call over the published vectors,
edge shapes and tampered records against client decryption, the plaintext word for word against the public-block path,
a message alone against the same message in the batch, and the descending-length prefix schedule under three keys."""
import numpy as np
import pytest

from conftest import SEED
from test_aes_multikey import RANDOM_KEY, assert_words_equal, schedule_cts

TAC_ERR_ARG, TAC_ERR_STATE = -2, -3

SP_KEY = bytes(range(0x40, 0x50))          # SP 800-38C Appendix C
RFC_KEY = bytes(range(0xC0, 0xD0))         # RFC 3610 §8

# (key, nonce, aad, plaintext, tag_len, C ‖ U)
VECTORS = {
    "sp800_38c_ex1": (SP_KEY, bytes(range(0x10, 0x17)), bytes(range(0x00, 0x08)), bytes(range(0x20, 0x24)), 4,
                      bytes.fromhex("7162015b4dac255d")),
    "sp800_38c_ex2": (SP_KEY, bytes(range(0x10, 0x18)), bytes(range(0x00, 0x10)), bytes(range(0x20, 0x30)), 6,
                      bytes.fromhex("d2a1f0e051ea5f62081a7792073d593d1fc64fbfaccd")),
    "sp800_38c_ex3": (SP_KEY, bytes(range(0x10, 0x1C)), bytes(range(0x00, 0x14)), bytes(range(0x20, 0x38)), 8,
                      bytes.fromhex("e3b201a9f5b71a7a9b1ceaeccd97e70b6176aad9a4428aa5484392fbc1b09951")),
    "rfc3610_packet1": (RFC_KEY, bytes.fromhex("00000003020100a0a1a2a3a4a5"), bytes(range(0x00, 0x08)), bytes(range(0x08, 0x1F)), 8,
                        bytes.fromhex("588c979a61c663d2f066d0c2c0f989806d5f6b61dac38417e8d12cfdf926e0")),
}


def aesccm(key, nonce, pt, tag_len, aad):
    from cryptography.hazmat.primitives.ciphers.aead import AESCCM
    return AESCCM(key, tag_length=tag_len).encrypt(nonce, pt, aad or None)


def ecb(key):
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    enc = Cipher(algorithms.AES(key), modes.ECB()).encryptor()
    return lambda block: enc.update(bytes(block))


def xor(a, b):
    return bytes(x ^ y for x, y in zip(a, b))


def ctr_plaintext(tac, key, nonce, data, tag_len, aad=b""):
    """what transciphering yields as plaintext, genuine or not: C ⊕ E(A_1 ‖ A_2 …) for the given nonce"""
    ctr, _ = tac.aes_ccm_format(nonce, data, tag_len, aad)
    E = ecb(key)
    p = len(data) - tag_len
    return xor(data[:p], b"".join(E(a) for a in ctr[1:]))


def replay(tac, key, nonce, pt, tag_len, aad):
    """AES-CCM encryption in clear AES from tac_aes_ccm_format's blocks: the plaintext goes into the zero payload blocks
    of the CBC-MAC sequence, which must be its last ceil(p/16) blocks"""
    ctr, mac = tac.aes_ccm_format(nonce, bytes(len(pt) + tag_len), tag_len, aad)
    m = (len(pt) + 15) // 16
    assert ctr.shape == (m + 1, 16)
    assert not mac[mac.shape[0] - m:].any()
    padded = np.frombuffer(pt + bytes(16 * m - len(pt)), dtype=np.uint8).reshape(m, 16)
    if m:
        mac[mac.shape[0] - m:] = padded
    E = ecb(key)
    x = E(mac[0])
    for blk in mac[1:]:
        x = E(xor(x, bytes(blk)))
    stream = [E(a) for a in ctr]
    return xor(pt, b"".join(stream[1:])) + xor(x[:tag_len], stream[0])


# ---------------------------------------------------------------------------------------------- formatting (host only)
@pytest.mark.parametrize("name", sorted(VECTORS))
def test_published_vectors(tac, name):
    key, nonce, aad, pt, t, want = VECTORS[name]
    assert aesccm(key, nonce, pt, t, aad) == want
    assert replay(tac, key, nonce, pt, t, aad) == want


AAD_LENGTHS = (0, 1, 13, 14, 65279, 65280, 70000)     # 65280 = 2^16 − 2^8: the 6-byte length prefix starts there
PAYLOAD_LENGTHS = (0, 1, 15, 16, 17, 100)
NONCE_LENGTHS = (7, 8, 12, 13)


def test_format_replays_aesccm(tac):
    """every nonce length × tag length at a small shape, and every AAD length × payload length with the nonce and tag
    lengths rotating, so that each value meets several of the others"""
    rng = np.random.default_rng(SEED)
    key = rng.bytes(16)
    cases = [(nl, t, 13, 17) for nl in NONCE_LENGTHS for t in tac.CCM_TAG_LENGTHS]
    cases += [(NONCE_LENGTHS[i % 4], tac.CCM_TAG_LENGTHS[i % 7], a, p)
              for i, (a, p) in enumerate((a, p) for a in AAD_LENGTHS for p in PAYLOAD_LENGTHS)]
    for nl, t, a, p in cases:
        nonce, aad, pt = rng.bytes(nl), rng.bytes(a), rng.bytes(p)
        assert replay(tac, key, nonce, pt, t, aad) == aesccm(key, nonce, pt, t, aad), (nl, t, a, p)


def test_format_blocks(tac):
    """B_0 flags and length, the AAD length prefix of each class, the counter blocks and the counts"""
    nonce = bytes(range(1, 13))
    ctr, mac = tac.aes_ccm_format(nonce, bytes(20 + 16), 16, b"")
    assert mac.shape == (3, 16) and ctr.shape == (3, 16)                 # no AAD: B_0 and two payload blocks
    assert bytes(mac[0]) == bytes([8 * 7 + 2]) + nonce + (20).to_bytes(3, "big")
    assert [bytes(c) for c in ctr] == [bytes([2]) + nonce + i.to_bytes(3, "big") for i in range(3)]
    for a, prefix in ((1, b"\x00\x01"), (65279, b"\xfe\xff"), (65280, b"\xff\xfe\x00\x00\xff\x00"), (70000, b"\xff\xfe" + (70000).to_bytes(4, "big"))):
        aad = bytes([0xA5]) * a
        _, mac = tac.aes_ccm_format(nonce, bytes(4), 4, aad)
        assert mac[0][0] == 64 + 8 + 2
        body = bytes(mac[1:].reshape(-1))
        assert mac.shape[0] == 1 + (len(prefix) + a + 15) // 16
        assert body[:len(prefix)] == prefix and body[len(prefix):len(prefix) + a] == aad and not any(body[len(prefix) + a:])


def test_argument_errors(tac):
    L = tac.load_library()
    counts = np.zeros(2, dtype=np.int64)

    def fmt(nonce_len=12, tag_len=16, aad_len=0, data_len=32, aad=True, data=True, nonce=True):
        buf = bytes(max(16, data_len, aad_len))
        m = tac.CcmMsg(tac.C.cast(tac.C.c_char_p(buf), tac.C.c_void_p).value if nonce else None, nonce_len, tag_len,
                       tac.C.cast(tac.C.c_char_p(buf), tac.C.c_void_p).value if aad else None, aad_len,
                       tac.C.cast(tac.C.c_char_p(buf), tac.C.c_void_p).value if data else None, data_len)
        return L.tac_aes_ccm_format(tac.C.addressof(m), None, None, counts.ctypes.data)

    assert fmt() == 0 and counts.tolist() == [2, 2]
    for bad in (dict(nonce_len=6), dict(nonce_len=14), dict(tag_len=5), dict(tag_len=2), dict(tag_len=18), dict(data_len=7, tag_len=8),
                dict(nonce_len=13, data_len=65536 + 16), dict(nonce=False), dict(aad=False, aad_len=1), dict(data=False)):
        assert fmt(**bad) == TAC_ERR_ARG, bad
    assert fmt(nonce_len=13, data_len=65535 + 16) == 0                 # q = 2 holds p < 2^16
    assert fmt(aad=False, aad_len=0) == 0
    assert L.tac_aes_ccm_format(None, None, None, counts.ctypes.data) == TAC_ERR_ARG
    bad_messages = [(bytes(6), bytes(20), 16, b""), (bytes(14), bytes(20), 16, b""), (bytes(12), bytes(20), 5, b""),
                    (bytes(12), bytes(20), 18, b""), (bytes(12), bytes(7), 8, b""), (bytes(13), bytes(65536 + 4), 4, b""),
                    (bytes(12), bytes(20), 16.0, b"")]
    for nonce, data, t, aad in bad_messages:
        with pytest.raises(ValueError):
            tac.aes_ccm_format(nonce, data, t, aad)
    # the context's checks run before any device call: this object has no device state at all
    ctx = object.__new__(tac.FheContext)
    ctx.L, ctx.params = L, tac.params_preset(64)
    ctx._n_keys = 2
    for nonce, data, t, aad in bad_messages:
        with pytest.raises(ValueError):
            ctx.aes_ccm_transcipher(nonce, data, t, aad)
        with pytest.raises(ValueError):
            ctx.aes_ccm_transcipher_many([(0, bytes(12), bytes(20), 16, b""), (1, nonce, data, t, aad)])
    for k in (-1, 2, 0.5):
        with pytest.raises(ValueError):
            ctx.aes_ccm_transcipher_many([(0, bytes(12), bytes(20), 16, b""), (k, bytes(12), bytes(20), 16, b"")])


# ---------------------------------------------------------------------------------------------- the device path
@pytest.fixture(scope="module")
def client(tac):
    """a second client on the session's lvl-64 secret keys (same seed) for this file's encryptions: the session client's
    encryption counter, which later tests' default-indexed encryptions follow, stays as it was"""
    return tac.ClientKey(64, seed=SEED)


def signed(x):
    return np.asarray(x, dtype=np.uint64).astype(np.int64).astype(np.float64)


def record(key, nonce, pt, t, aad):
    return dict(key=key, nonce=nonce, aad=aad, t=t, data=aesccm(key, nonce, pt, t, aad), pt=pt, genuine=True)


def flip(b, bit):
    b = bytearray(b)
    b[bit // 8] ^= 0x80 >> (bit % 8)
    return bytes(b)


def batch_records():
    """the published vectors, edge shapes and four tampered records, two keys (0: SP_KEY, 1: RFC_KEY)"""
    rng = np.random.default_rng(SEED + 1)
    recs = []
    for name in sorted(VECTORS):
        key, nonce, aad, pt, t, _ = VECTORS[name]
        recs.append(record(key, nonce, pt, t, aad))
    recs.append(record(RFC_KEY, rng.bytes(12), b"", 16, rng.bytes(13)))                         # AAD only
    recs.append(record(SP_KEY, rng.bytes(13), rng.bytes(40), 4, b""))                            # no AAD, tag 4
    recs.append(record(RFC_KEY, rng.bytes(8), b"", 8, b""))                                      # no chain step at all
    base = record(RFC_KEY, rng.bytes(12), rng.bytes(37), 16, rng.bytes(13))
    ct_flip = dict(base, data=flip(base["data"], 21), pt=flip(base["pt"], 21), genuine=False)    # flipped ciphertext bit
    tag = record(SP_KEY, rng.bytes(12), rng.bytes(20), 12, rng.bytes(5))
    tag_flip = dict(tag, data=flip(tag["data"], 8 * 20 + 3), genuine=False)                      # flipped tag bit
    aad = record(RFC_KEY, rng.bytes(7), rng.bytes(16), 16, rng.bytes(30))
    aad_alt = dict(aad, aad=flip(aad["aad"], 9), genuine=False)                                  # altered AAD
    nonce = record(SP_KEY, rng.bytes(11), rng.bytes(33), 10, rng.bytes(3))
    nonce_alt = dict(nonce, nonce=flip(nonce["nonce"], 0), genuine=False)                        # wrong nonce
    return recs + [ct_flip, tag_flip, aad_alt, nonce_alt]


def key_index(rec, keys):
    return keys.index(rec["key"])


@pytest.mark.gpu
def test_batched_records_and_tampering(tac, gpu64, client, ol):
    ck, ctx = client, gpu64[1]
    L1 = ck.params.big_lwe_size
    keys = [SP_KEY, RFC_KEY]
    scheds = schedule_cts(ck, ol, keys, 1 << 52)
    ctx.aes_set_key_table(scheds)
    recs = batch_records()
    msgs = [(key_index(r, keys), r["nonce"], r["data"], r["t"], r["aad"]) for r in recs]
    out = ctx.aes_ccm_transcipher_many(msgs)
    assert len(out) == len(recs)
    worst = 0.0
    for i, (r, (pt, valid)) in enumerate(zip(recs, out)):
        p = len(r["data"]) - r["t"]
        assert pt.shape == (p, 8, L1) and valid.shape == (L1,), i
        want_pt = ctr_plaintext(tac, r["key"], r["nonce"], r["data"], r["t"], r["aad"])
        if i != len(recs) - 1:                                          # all but the wrong nonce decrypt to their payload
            assert want_pt == r["pt"], i
        assert ck.decrypt_bytes(pt) == want_pt, i
        bit = int(ck.decrypt_bits(valid)[0])
        assert bit == int(r["genuine"]), (i, bit)
        worst = max(worst, float(np.abs(signed(ck.decrypt_phases(valid) - (np.uint64(bit) << np.uint64(63)))).max()))
        # the plaintext bits are the public-block path's words over the same counter blocks with XOR bytes C
        ctr, _ = tac.aes_ccm_format(r["nonce"], r["data"], r["t"], r["aad"])
        if p:
            m = ctr.shape[0] - 1
            ref = ctx.aes_encrypt_public_blocks_keyed(ctr[1:], [msgs[i][0]] * m, xor=r["data"][:p] + bytes(16 * m - p))
            assert_words_equal(pt, ref.reshape(-1, 8, L1)[:p], f"record {i} against aes_encrypt_public_blocks_keyed")
    print(f"largest validity-bit phase error: 2^{np.log2(worst + 1):.1f}")
    assert worst < 2.0 ** 59
    # a record alone gives the words it got in the batch, keyed and under the single schedule
    for i in (2, 3, 8, 9):
        r = recs[i]
        (pt, valid), = ctx.aes_ccm_transcipher_many([msgs[i]])
        assert_words_equal(pt, out[i][0], f"record {i} alone, plaintext")
        assert_words_equal(valid[None], out[i][1][None], f"record {i} alone, validity bit")
    ctx.aes_set_key_schedule(scheds[1])
    r = recs[0]
    assert r["key"] == RFC_KEY
    pt, valid = ctx.aes_ccm_transcipher(r["nonce"], r["data"], r["t"], r["aad"])
    assert_words_equal(pt, out[0][0], "RFC 3610 packet 1 under the single schedule, plaintext")
    assert_words_equal(valid[None], out[0][1][None], "RFC 3610 packet 1 under the single schedule, validity bit")


@pytest.mark.gpu
def test_prefix_schedule_under_three_keys(tac, gpu64, client, ol):
    """chain lengths 0..6 interleaved over three table entries: the internal descending-length order must give every
    message the words of its own single-key run"""
    ck, ctx = client, gpu64[1]
    keys = [SP_KEY, RFC_KEY, RANDOM_KEY]
    scheds = schedule_cts(ck, ol, keys, 1 << 53)
    ctx.aes_set_key_table(scheds)
    rng = np.random.default_rng(SEED + 2)
    shapes = [(2, 1, 30), (0, 13, 80), (1, 0, 0), (2, 40, 17), (0, 0, 16), (1, 13, 40), (2, 0, 20)]   # key, |A|, p
    recs = []
    for i, (k, a, p) in enumerate(shapes):
        r = record(keys[k], rng.bytes(12), rng.bytes(p), 16, rng.bytes(a))
        recs.append(dict(r, data=flip(r["data"], 8 * p + 1)) if i == 3 else r)               # one bad tag in the mix
    chains = [tac.aes_ccm_format(r["nonce"], r["data"], 16, r["aad"])[1].shape[0] - 1 for r in recs]
    assert chains == [3, 6, 0, 5, 1, 4, 2], chains
    out = ctx.aes_ccm_transcipher_many([(k, r["nonce"], r["data"], 16, r["aad"]) for (k, _, _), r in zip(shapes, recs)])
    for i, ((k, _, _), r, (pt, valid)) in enumerate(zip(shapes, recs, out)):
        assert ck.decrypt_bytes(pt) == r["pt"], i
        assert int(ck.decrypt_bits(valid)[0]) == (i != 3), i
        ctx.aes_set_key_schedule(scheds[k])
        spt, svalid = ctx.aes_ccm_transcipher(r["nonce"], r["data"], 16, r["aad"])
        assert_words_equal(pt, spt, f"message {i}: plaintext against its single-key run")
        assert_words_equal(valid[None], svalid[None], f"message {i}: validity bit against its single-key run")


@pytest.mark.gpu
def test_state_and_argument_errors(tac, ck64):
    ctx = tac.FheContext(ck64.params, device=0)                # no keys, no schedule, no table
    L = ctx.L
    nonce, data = bytes(12), bytes(32)
    msgs, keep, _ = tac._ccm_messages([(nonce, data, 16, b"")])
    L1 = ck64.params.big_lwe_size
    pt, valid = np.zeros((16, 8, L1), dtype=np.uint64), np.zeros(L1, dtype=np.uint64)
    kidx = np.zeros(1, dtype=np.int32)
    assert L.tac_aes_ccm_transcipher(ctx.h, 1, None, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_STATE
    assert L.tac_aes_ccm_transcipher(ctx.h, 1, kidx.ctypes.data, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_STATE
    assert L.tac_aes_ccm_transcipher(ctx.h, -1, None, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_ARG
    assert L.tac_aes_ccm_transcipher(ctx.h, 1, None, None, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_ARG
    bad, keep2, _ = tac._ccm_messages([(nonce, data, 16, b"")])
    bad[0].tag_len = 5
    assert L.tac_aes_ccm_transcipher_dev(ctx.h, 1, None, bad, None, None) == TAC_ERR_ARG
    ctx.upload_keys(ck64)
    ctx.aes_set_key_table(np.zeros((2, 44, 4, 8, L1), dtype=np.uint64))
    launches = ctx.launch_count()
    assert L.tac_aes_ccm_transcipher(ctx.h, 0, kidx.ctypes.data, None, None, None) == 0
    for k in (-1, 2):
        kidx[0] = k
        assert L.tac_aes_ccm_transcipher(ctx.h, 1, kidx.ctypes.data, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_ARG
    assert "outside [0, 2)" in ctx.last_error()
    kidx[0] = 0
    assert L.tac_aes_ccm_transcipher(ctx.h, 1, kidx.ctypes.data, msgs, pt.ctypes.data, None) == TAC_ERR_ARG
    assert L.tac_aes_ccm_transcipher(ctx.h, 1, None, msgs, pt.ctypes.data, valid.ctypes.data) == TAC_ERR_STATE   # no single schedule
    assert ctx.launch_count() == launches
    # params_sqrd_lvl_4 cannot hold a middle round's 33: NoiseTooBig before anything else is looked at
    small = tac.FheContext(4, device=0)
    with pytest.raises(tac.NoiseTooBig):
        small.aes_ccm_transcipher(nonce, data)
