#!/usr/bin/env python
"""decrypt_bench.py — AES-128 decryption on one B200 next to encryption, and AES-CBC transciphering.

    python tools/decrypt_bench.py [--blocks 128] [--steps 3] [--warmup 1] [--device 0]

All arms run 10 rounds over N blocks under the CLI key.  The key schedule comes from the device key expansion of the
FHE-encrypted key; the inverse key schedule dk is derived from it on the device (tac_aes_inv_key_schedule, timed once
after one warm-up call and decrypt-checked against the clear InvMixColumns schedule).
  encrypt         tac_aes_encrypt_blocks_dev on FHE-encrypted random blocks, inputs resident in HBM (bench.py's step)
  decrypt         tac_aes_decrypt_blocks_dev on the encrypt arm's output (squared noise 9): the round trip is its check
  cbc_transcipher tac_aes_decrypt_public_blocks_dev on an N-block AES-CBC ciphertext with the previous ciphertext blocks
                  (IV first) as XOR bytes: FHE encryptions of the plaintext
Timed steps alternate between the arms, each timed with CUDA events on the context's stream.  Every arm's output is
decrypted and checked against clear AES.  Prints one JSON line with the card's name and power limit.
"""
import argparse
import importlib
import json
import os
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from bench import CLI_KEY, SEED, clear_aes, clear_key_schedule  # noqa: E402
from ctr_bench import gpu_info  # noqa: E402


def clear_inv_key_schedule(ek):
    """dk of the equivalent inverse cipher from the 176-byte schedule: InvMixColumns on round keys 1..9"""
    def mul(a, b):
        r = 0
        for _ in range(8):
            if b & 1:
                r ^= a
            a = ((a << 1) ^ (0x1B if a & 0x80 else 0)) & 0xFF
            b >>= 1
        return r
    coef = (14, 11, 13, 9)
    dk = bytearray(ek)
    for q in range(4, 40):                   # words of round keys 1..9
        col = ek[4 * q:4 * q + 4]
        dk[4 * q:4 * q + 4] = bytes(
            mul(col[0], coef[-r & 3]) ^ mul(col[1], coef[(1 - r) & 3]) ^ mul(col[2], coef[(2 - r) & 3]) ^ mul(col[3], coef[(3 - r) & 3])
            for r in range(4))
    return bytes(dk)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=128)
    ap.add_argument("--steps", type=int, default=3, help="timed steps per arm (alternating)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    if args.blocks < 1 or args.steps < 1 or args.warmup < 0:
        ap.error("--blocks and --steps must be >= 1, --warmup >= 0")

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("decrypt_bench.py needs a CUDA device")
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    tac = importlib.import_module("tfhe-aes-2_b200")
    device = torch.device("cuda", args.device)
    torch.cuda.set_device(device)
    stream = torch.cuda.current_stream(device)

    ck = tac.ClientKey(64, seed=SEED).gen_eval_keys()
    ctx = tac.FheContext(ck.params, device=args.device, stream=stream.cuda_stream)
    ctx.upload_keys(ck)
    L1, nb = ck.params.big_lwe_size, args.blocks
    ks = ctx.aes_key_schedule(ck.encrypt_bytes(CLI_KEY, first_index=1 << 40))
    ok_ks = ck.decrypt_bytes(ks.reshape(-1, L1)) == clear_key_schedule(CLI_KEY)

    # inverse key schedule: one warm-up call (registers the decryption LUTs), then one timed call
    ctx._check(ctx.L.tac_aes_inv_key_schedule(ctx.h, None))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    ctx._check(ctx.L.tac_aes_inv_key_schedule(ctx.h, None))
    e1.record(stream)
    torch.cuda.synchronize(device)
    inv_ks_ms = e0.elapsed_time(e1)
    dk = ctx.aes_inv_key_schedule()
    ok_dk = ck.decrypt_bytes(dk.reshape(-1, L1)) == clear_inv_key_schedule(clear_key_schedule(CLI_KEY))

    rng = np.random.default_rng(SEED)
    plain = [rng.bytes(16) for _ in range(nb)]
    in_np = np.stack([ck.encrypt_bytes(b, first_index=(1 + i) * 128) for i, b in enumerate(plain)])
    in_dev = torch.from_numpy(in_np.view(np.int64)).to(device)
    out_enc = torch.empty_like(in_dev)
    out_dec = torch.empty_like(in_dev)
    out_cbc = torch.empty_like(in_dev)

    iv = rng.bytes(16)
    msg = rng.bytes(16 * nb)
    ct = Cipher(algorithms.AES(CLI_KEY), modes.CBC(iv)).encryptor().update(msg)
    cbc_blocks = np.frombuffer(ct, dtype=np.uint8).reshape(nb, 16)
    cbc_xor = np.frombuffer(iv + ct[:-16], dtype=np.uint8).reshape(nb, 16)
    plan = tac.aes_public_plan(cbc_blocks, decrypt=True)

    arms = {
        "encrypt": lambda: ctx.aes_encrypt_blocks_dev(nb, in_dev.data_ptr(), out_enc.data_ptr()),
        "decrypt": lambda: ctx.aes_decrypt_blocks_dev(nb, out_enc.data_ptr(), out_dec.data_ptr(), in_noise_sq=9),
        "cbc_transcipher": lambda: ctx.aes_decrypt_public_blocks_dev(cbc_blocks, out_cbc.data_ptr(), xor=cbc_xor),
    }
    for _ in range(args.warmup):
        for run in arms.values():
            run()
    torch.cuda.synchronize(device)
    ms = {k: [] for k in arms}
    for _ in range(args.steps):
        for name, run in arms.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            run()
            e1.record(stream)
            torch.cuda.synchronize(device)
            ms[name].append(e0.elapsed_time(e1))

    enc = out_enc.cpu().numpy().view(np.uint64)
    dec = out_dec.cpu().numpy().view(np.uint64)
    cbc = out_cbc.cpu().numpy().view(np.uint64)
    ok_enc = all(ck.decrypt_bytes(enc[i]) == clear_aes(CLI_KEY, plain[i]) for i in range(nb))
    ok_dec = all(ck.decrypt_bytes(dec[i]) == plain[i] for i in range(nb))
    ok_cbc = ck.decrypt_bytes(cbc) == msg

    info = gpu_info(args.device)
    rate = {k: nb / (np.mean(v) * 1e-3) for k, v in ms.items()}
    line = {
        "metric": "fhe_aes128_decrypt_blocks_per_s", "unit": "blocks/s", "blocks": nb, "rounds": 10,
        "steps": args.steps, "warmup": args.warmup, "parameter_set": "params_sqrd_lvl_64 (n=677,k=4,N=512)",
        "encrypt": {"value": rate["encrypt"], "ms_per_step": ms["encrypt"], "boxes_per_round": [16 * nb] * 10},
        "decrypt": {"value": rate["decrypt"], "ms_per_step": ms["decrypt"], "boxes_per_round": [16 * nb] * 10},
        "cbc_transcipher": {"value": rate["cbc_transcipher"], "ms_per_step": ms["cbc_transcipher"], "boxes_per_round": plan},
        "decrypt_over_encrypt": rate["decrypt"] / rate["encrypt"],
        "inv_key_schedule_ms": inv_ks_ms,
        "gpu": info,
        "verified": {"key_schedule": ok_ks, "inv_key_schedule": ok_dk, "encrypt": ok_enc, "decrypt": ok_dec, "cbc_transcipher": ok_cbc},
    }
    print(json.dumps(line), flush=True)
    if not all(line["verified"].values()):
        raise SystemExit("decrypt_bench: check FAILED")


if __name__ == "__main__":
    main()
