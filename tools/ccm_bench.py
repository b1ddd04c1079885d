#!/usr/bin/env python
"""ccm_bench.py — AES-CCM transciphering with the tag checked under FHE, against unauthenticated CTR transciphering of
the same payloads, on one B200.

    python tools/ccm_bench.py [--records 128] [--steps 2] [--warmup 1] [--device 0] [--out profiles/ccm_bench_128records.json]

Workload: --records TLS-1.2-shaped AES-CCM records (12-byte nonce, 13-byte AAD, 64-byte payload, 16-byte tag), record i
under key table entry i (random keys, expanded on the device with tac_aes_key_table); every 16th record has one flipped
tag bit.  params_sqrd_lvl_64, 10-round AES-128.  Timed steps alternate between the two arms, each timed on the host around
a host-buffer call (copies included) that ends in a device synchronisation:
  a  aes_ccm_transcipher_many: plaintext bits and an encrypted validity bit per record
  b  the CTR half alone: aes_encrypt_public_blocks_keyed over the same records' CCM counter blocks A_1..A_4 with XOR bytes
     C, i.e. what aes_ctr_transcipher_many runs for CTR counter blocks (the unauthenticated baseline)
Circuit bootstraps per arm: the planner's count for the public-block call (tac_aes_public_plan_keyed) plus, for arm a,
160 per CBC-MAC chain block and 19 per record for the tag check.  Every output is checked by client decryption: the
plaintext against `cryptography`'s AESCCM, the validity bit 0 for the tampered records and 1 for the rest.  Writes one JSON
line with the card's name and power limit to --out and prints it.
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

NONCE, AAD, PAYLOAD, TAG = 12, 13, 64, 16
TAMPER_EVERY = 16
TAG_CHECK_BOXES = 19            # 16 byte-zero tests, 2 eight-bit ANDs, 1 two-bit AND
BOXES_PER_BLOCK = 160           # 10 rounds × 16 S-boxes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=128, help="records, each under its own key table entry")
    ap.add_argument("--steps", type=int, default=2, help="timed steps per arm (alternating)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "ccm_bench_128records.json"))
    args = ap.parse_args()
    if args.records < 1 or args.steps < 1 or args.warmup < 0:
        ap.error("--records >= 1, --steps >= 1, --warmup >= 0")

    import torch
    from cryptography.hazmat.primitives.ciphers.aead import AESCCM
    if not torch.cuda.is_available():
        raise SystemExit("ccm_bench.py needs a CUDA device")
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
    recs = []
    for i in range(n):
        nonce, aad, pt = rng.bytes(NONCE), rng.bytes(AAD), rng.bytes(PAYLOAD)
        data = AESCCM(keys[i], tag_length=TAG).encrypt(nonce, pt, aad)
        tampered = i % TAMPER_EVERY == TAMPER_EVERY - 1
        if tampered:
            data = data[:PAYLOAD] + bytes([data[PAYLOAD] ^ 0x10]) + data[PAYLOAD + 1:]
        recs.append(dict(nonce=nonce, aad=aad, pt=pt, data=data, tampered=tampered))
    key_bits = np.stack([ck.encrypt_bytes(k, first_index=(1 << 40) + 128 * i) for i, k in enumerate(keys)])
    ctx.aes_key_table(key_bits)                       # the resident key table (its host copy is dropped)

    msgs = [(i, r["nonce"], r["data"], TAG, r["aad"]) for i, r in enumerate(recs)]
    fmt = [tac.aes_ccm_format(r["nonce"], r["data"], TAG, r["aad"]) for r in recs]
    m = fmt[0][0].shape[0] - 1                         # payload blocks per record
    chain = fmt[0][1].shape[0] - 1                     # CBC-MAC blocks after B_0 per record
    ctr_blocks = np.concatenate([c[1:] for c, _ in fmt])
    ctr_kidx = np.repeat(np.arange(n), m)
    ctr_xor = b"".join(r["data"][:PAYLOAD] for r in recs)
    # arm a's public call: [B_0 rows][A_0 rows][A_1..A_m rows]; the records all have the same chain length, so the
    # descending-length order is the records' own
    pub_blocks = np.concatenate([np.stack([mac[0] for _, mac in fmt]), np.stack([c[0] for c, _ in fmt]), ctr_blocks])
    pub_kidx = np.concatenate([np.arange(n), np.arange(n), ctr_kidx])
    boxes_a_public = sum(tac.aes_public_plan(pub_blocks, key_index=pub_kidx))
    boxes_b = sum(tac.aes_public_plan(ctr_blocks, key_index=ctr_kidx))
    boxes_a = boxes_a_public + BOXES_PER_BLOCK * chain * n + TAG_CHECK_BOXES * n

    res = {}
    arms = {
        "a_ccm": lambda: res.__setitem__("a", ctx.aes_ccm_transcipher_many(msgs)),
        "b_ctr": lambda: res.__setitem__("b", ctx.aes_encrypt_public_blocks_keyed(ctr_blocks, ctr_kidx, xor=ctr_xor)),
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

    valid = [int(ck.decrypt_bits(v)[0]) for _, v in res["a"]]
    b_pt = res["b"].reshape(n, m * 16, 8, -1)
    verified = {
        "a_plaintext": all(ck.decrypt_bytes(pt) == r["pt"] for (pt, _), r in zip(res["a"], recs)),
        "a_validity": valid == [int(not r["tampered"]) for r in recs],
        "b_plaintext": all(ck.decrypt_bytes(b_pt[i][:PAYLOAD]) == r["pt"] for i, r in enumerate(recs)),
    }
    identical = all(np.array_equal(pt, b_pt[i][:PAYLOAD]) for i, (pt, _) in enumerate(res["a"]))

    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    rate = {k: n / (mean[k] * 1e-3) for k in ms}
    ratio = boxes_a / boxes_b
    predicted_a = rate["b_ctr"] / ratio
    line = {
        "metric": "fhe_aes128_ccm_transcipher", "records": n, "keys": n, "nonce_bytes": NONCE, "aad_bytes": AAD,
        "payload_bytes": PAYLOAD, "tag_bytes": TAG, "tampered": sum(r["tampered"] for r in recs), "rounds": 10,
        "steps": args.steps, "warmup": args.warmup, "parameter_set": "params_sqrd_lvl_64 (n=677,k=4,N=512)",
        "a_ccm": {"records_per_s": rate["a_ccm"], "payload_bytes_per_s": rate["a_ccm"] * PAYLOAD, "boxes": boxes_a,
                  "boxes_public_call": boxes_a_public, "chain_blocks": chain * n, "boxes_tag_check": TAG_CHECK_BOXES * n},
        "b_ctr": {"records_per_s": rate["b_ctr"], "payload_bytes_per_s": rate["b_ctr"] * PAYLOAD, "boxes": boxes_b},
        "box_ratio": ratio, "a_predicted_records_per_s": predicted_a, "a_vs_prediction": rate["a_ccm"] / predicted_a,
        "ms_per_step": ms, "gpu": gpu_info(args.device), "verified": verified, "plaintext_identical": identical,
    }
    text = json.dumps(line)
    print(text, flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
    if not (all(verified.values()) and identical):
        raise SystemExit("ccm_bench: check FAILED")


if __name__ == "__main__":
    main()
