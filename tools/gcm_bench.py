#!/usr/bin/env python
"""gcm_bench.py — AES-GCM transciphering with the tag checked under FHE, against its unauthenticated CTR half and against
AES-CCM transciphering of same-shaped records, on one B200.

    python tools/gcm_bench.py [--records 128] [--steps 2] [--warmup 1] [--depth 8] [--device 0] [--out profiles/gcm_bench_128records.json]

Workload: the TLS-shaped records of ccm_bench.py (12-byte IV / nonce, 13-byte AAD, 64-byte payload, 16-byte tag), record i
under key table entry i (random keys, expanded on the device with tac_aes_key_table); every 16th record has one flipped tag
bit.  params_sqrd_lvl_64, 10-round AES-128.  The 128-key GHASH key table (depth --depth) is built once and timed on its own.
Timed steps alternate between three arms, each timed on the host around a host-buffer call that ends in a device
synchronisation:
  a  aes_gcm_transcipher_many: plaintext bits and an encrypted validity bit per record (M = 6 GHASH blocks <= depth: no
     encrypted GF(2^128) product)
  b  the CTR half alone: aes_encrypt_public_blocks_keyed over the same records' counter blocks inc32^i(J0) with XOR bytes C
  c  aes_ccm_transcipher_many over AES-CCM records of the same shape under the same keys
Circuit bootstraps per arm: the planner's count for the public-block calls (tac_aes_public_plan_keyed); for arm a plus the
GHASH refreshes (one per run of at most max_noise_level_squared terms of one GHASH block in a tag-difference bit, the
planner's first level) and 19 per record for the tag check; for arm c plus 160 per CBC-MAC block and 19 per record.  Every
output is checked by client decryption against `cryptography`'s AESGCM / AESCCM.  Writes one JSON line with the card's
name and power limit to --out and prints it.
"""
import argparse
import importlib
import json
import os
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import numpy as np  # noqa: E402

from bench import SEED  # noqa: E402
from ctr_bench import gpu_info  # noqa: E402

IV, AAD, PAYLOAD, TAG = 12, 13, 64, 16
TAMPER_EVERY = 16
TAG_CHECK_BOXES = 19            # 16 byte-zero tests, 2 eight-bit ANDs, 1 two-bit AND
BOXES_PER_BLOCK = 160           # 10 rounds × 16 S-boxes
MAX_NOISE = 64                  # params_sqrd_lvl_64


def ghash_refreshes(blocks, t):
    """refreshes of the linear layer of a record of at most depth blocks: for each of the 8t tag-difference bits and each
    block X_i, its terms (bit j of X_i · x^l over l, squared noise 1 each) in runs of at most MAX_NOISE"""
    total = 0
    for b in blocks:
        col, count = int.from_bytes(bytes(b), "big"), [0] * (8 * t)
        for _ in range(128):
            for j in range(8 * t):
                count[j] += (col >> (127 - j)) & 1
            col = (col >> 1) ^ (0xE1 << 120) if col & 1 else col >> 1         # times x (SP 800-38D)
        total += sum((c + MAX_NOISE - 1) // MAX_NOISE for c in count if c > 1)
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=128, help="records, each under its own key table entry")
    ap.add_argument("--steps", type=int, default=2, help="timed steps per arm (alternating)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--depth", type=int, default=8, help="powers of H in the GHASH key table")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "gcm_bench_128records.json"))
    args = ap.parse_args()
    if args.records < 1 or args.steps < 1 or args.warmup < 0:
        ap.error("--records >= 1, --steps >= 1, --warmup >= 0")

    import torch
    from cryptography.hazmat.primitives.ciphers.aead import AESCCM, AESGCM
    if not torch.cuda.is_available():
        raise SystemExit("gcm_bench.py needs a CUDA device")
    tac = importlib.import_module("tfhe-aes-2_b200")
    device = torch.device("cuda", args.device)
    torch.cuda.set_device(device)
    stream = torch.cuda.current_stream(device)

    ck = tac.ClientKey(64, seed=SEED).gen_eval_keys()
    ctx = tac.FheContext(ck.params, device=args.device, stream=stream.cuda_stream)
    ctx.upload_keys(ck)
    n = args.records
    rng = np.random.default_rng(SEED)
    keys = [rng.bytes(16) for _ in range(n)]
    gcm, ccm = [], []
    for i in range(n):
        iv, aad, pt = rng.bytes(IV), rng.bytes(AAD), rng.bytes(PAYLOAD)
        tampered = i % TAMPER_EVERY == TAMPER_EVERY - 1
        for recs, data in ((gcm, AESGCM(keys[i]).encrypt(iv, pt, aad)), (ccm, AESCCM(keys[i], tag_length=TAG).encrypt(iv, pt, aad))):
            if tampered:
                data = data[:PAYLOAD] + bytes([data[PAYLOAD] ^ 0x10]) + data[PAYLOAD + 1:]
            recs.append(dict(iv=iv, aad=aad, pt=pt, data=data, tampered=tampered))
    key_bits = np.stack([ck.encrypt_bytes(k, first_index=(1 << 40) + 128 * i) for i, k in enumerate(keys)])
    ctx.aes_key_table(key_bits)
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    ctx.aes_gcm_hash_key_table(args.depth)
    table_s = time.perf_counter() - t0

    gcm_msgs = [(i, r["iv"], r["data"], TAG, r["aad"]) for i, r in enumerate(gcm)]
    ccm_msgs = [(i, r["iv"], r["data"], TAG, r["aad"]) for i, r in enumerate(ccm)]
    fmt = [tac.aes_gcm_format(r["iv"], r["data"], TAG, r["aad"]) for r in gcm]
    m, M = fmt[0][0].shape[0] - 1, fmt[0][1].shape[0]
    if M > args.depth:
        raise SystemExit(f"records of {M} GHASH blocks exceed --depth {args.depth}")
    ctr_blocks = np.concatenate([c[1:] for c, _ in fmt])
    ctr_kidx = np.repeat(np.arange(n), m)
    ctr_xor = b"".join(r["data"][:PAYLOAD] for r in gcm)
    boxes_b = sum(tac.aes_public_plan(ctr_blocks, key_index=ctr_kidx))
    boxes_a_public = sum(tac.aes_public_plan(np.concatenate([np.stack([c[0] for c, _ in fmt]), ctr_blocks]),
                                             key_index=np.concatenate([np.arange(n), ctr_kidx])))
    boxes_a_ghash = sum(ghash_refreshes(x, TAG) for _, x in fmt)
    boxes_a = boxes_a_public + boxes_a_ghash + TAG_CHECK_BOXES * n
    cfmt = [tac.aes_ccm_format(r["iv"], r["data"], TAG, r["aad"]) for r in ccm]
    c_ctr = np.concatenate([c[1:] for c, _ in cfmt])
    chain = cfmt[0][1].shape[0] - 1
    boxes_c = (sum(tac.aes_public_plan(np.concatenate([np.stack([mac[0] for _, mac in cfmt]), np.stack([c[0] for c, _ in cfmt]), c_ctr]),
                                       key_index=np.concatenate([np.arange(n), np.arange(n), np.repeat(np.arange(n), m)])))
               + BOXES_PER_BLOCK * chain * n + TAG_CHECK_BOXES * n)

    res = {}
    arms = {
        "a_gcm": lambda: res.__setitem__("a", ctx.aes_gcm_transcipher_many(gcm_msgs)),
        "b_ctr": lambda: res.__setitem__("b", ctx.aes_encrypt_public_blocks_keyed(ctr_blocks, ctr_kidx, xor=ctr_xor)),
        "c_ccm": lambda: res.__setitem__("c", ctx.aes_ccm_transcipher_many(ccm_msgs)),
    }
    for _ in range(args.warmup):
        for run in arms.values():
            run()
    torch.cuda.synchronize(device)
    ms = {k: [] for k in arms}
    for _ in range(args.steps):
        for name, run in arms.items():
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            run()
            torch.cuda.synchronize(device)
            ms[name].append((time.perf_counter() - t0) * 1e3)

    b_pt = res["b"].reshape(n, m * 16, 8, -1)
    verified = {
        "a_plaintext": all(ck.decrypt_bytes(pt) == r["pt"] for (pt, _), r in zip(res["a"], gcm)),
        "a_validity": [int(ck.decrypt_bits(v)[0]) for _, v in res["a"]] == [int(not r["tampered"]) for r in gcm],
        "b_plaintext": all(ck.decrypt_bytes(b_pt[i][:PAYLOAD]) == r["pt"] for i, r in enumerate(gcm)),
        "c_plaintext": all(ck.decrypt_bytes(pt) == r["pt"] for (pt, _), r in zip(res["c"], ccm)),
        "c_validity": [int(ck.decrypt_bits(v)[0]) for _, v in res["c"]] == [int(not r["tampered"]) for r in ccm],
    }
    identical = all(np.array_equal(pt, b_pt[i][:PAYLOAD]) for i, (pt, _) in enumerate(res["a"]))

    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    rate = {k: n / (mean[k] * 1e-3) for k in ms}
    boxes = {"a_gcm": boxes_a, "b_ctr": boxes_b, "c_ccm": boxes_c}
    line = {
        "metric": "fhe_aes128_gcm_transcipher", "records": n, "keys": n, "iv_bytes": IV, "aad_bytes": AAD,
        "payload_bytes": PAYLOAD, "tag_bytes": TAG, "ghash_blocks": M, "depth": args.depth,
        "tampered": sum(r["tampered"] for r in gcm), "rounds": 10, "steps": args.steps, "warmup": args.warmup,
        "parameter_set": "params_sqrd_lvl_64 (n=677,k=4,N=512)", "hash_key_table_s": table_s,
        **{k: {"records_per_s": rate[k], "payload_bytes_per_s": rate[k] * PAYLOAD, "boxes": boxes[k],
               "predicted_records_per_s": rate["b_ctr"] * boxes_b / boxes[k], "vs_prediction": rate[k] / (rate["b_ctr"] * boxes_b / boxes[k])}
           for k in arms},
        "a_boxes_public_call": boxes_a_public, "a_boxes_ghash_refreshes": boxes_a_ghash, "a_boxes_tag_check": TAG_CHECK_BOXES * n,
        "ms_per_step": ms, "gpu": gpu_info(args.device), "verified": verified, "plaintext_identical": identical,
    }
    text = json.dumps(line)
    print(text, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
    if not (all(verified.values()) and identical):
        raise SystemExit("gcm_bench: check FAILED")


if __name__ == "__main__":
    main()
