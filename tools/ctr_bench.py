#!/usr/bin/env python
"""ctr_bench.py — AES-CTR keystream on one B200: encrypted counter blocks vs public counter blocks.

    python tools/ctr_bench.py [--blocks 128] [--steps 3] [--warmup 1] [--device 0]

Both arms run 10-round AES-128 over the counter blocks iv ‖ BE64(ctr), ctr = 1..N, under the CLI key and IV, with the key
schedule precomputed (as bench.py does):
  encrypted  tac_aes_encrypt_blocks_dev on FHE-encrypted counter blocks, inputs resident in HBM (bench.py's step)
  public     tac_aes_encrypt_public_blocks_dev on the clear counter blocks; S-box circuit bootstraps whose inputs are equal
             across blocks run once (aes_public_plan gives the count per round)
Timed steps alternate between the arms, each timed with CUDA events on the context's stream.  Both outputs are decrypted
and checked against clear AES; the public output must also equal, word for word, the encrypted path fed trivial
ciphertexts of the same blocks.  One host-buffer transcipher of N·16 bytes (tac_aes_encrypt_public_blocks with the XOR
bytes, copies included) is timed as well.  Prints one JSON line.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from bench import CLI_IV, CLI_KEY, SEED, clear_aes, clear_key_schedule  # noqa: E402


def gpu_info(index):
    """name and power limit of the card (read-only query)"""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", str(index)],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"name": out[0], "power_limit_w": float(out[1]), "sm_max_mhz": float(out[2])}
    except Exception:
        import torch
        return {"name": torch.cuda.get_device_name(index), "power_limit_w": None, "sm_max_mhz": None}


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
        raise SystemExit("ctr_bench.py needs a CUDA device")
    tac = importlib.import_module("tfhe-aes-2_b200")
    device = torch.device("cuda", args.device)
    torch.cuda.set_device(device)
    stream = torch.cuda.current_stream(device)

    ck = tac.ClientKey(64, seed=SEED).gen_eval_keys()
    ctx = tac.FheContext(ck.params, device=args.device, stream=stream.cuda_stream)
    ctx.upload_keys(ck)
    ctx.aes_set_key_schedule(ck.encrypt_bytes(clear_key_schedule(CLI_KEY), first_index=1 << 40))
    L1, nb = ck.params.big_lwe_size, args.blocks
    blocks = tac.ctr_blocks(CLI_IV, 1, nb)
    clear = [clear_aes(CLI_KEY, bytes(b)) for b in blocks]
    plan = tac.aes_public_plan(blocks)

    in_np = np.stack([ck.encrypt_bytes(bytes(b), first_index=(1 + i) * 128) for i, b in enumerate(blocks)])
    in_dev = torch.from_numpy(in_np.view(np.int64)).to(device)
    out_enc = torch.empty_like(in_dev)
    out_pub = torch.empty_like(in_dev)

    arms = {
        "encrypted": lambda: ctx.aes_encrypt_blocks_dev(nb, in_dev.data_ptr(), out_enc.data_ptr()),
        "public": lambda: ctx.aes_encrypt_public_blocks_dev(blocks, out_pub.data_ptr()),
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
    pub = out_pub.cpu().numpy().view(np.uint64)
    ok_enc = all(ck.decrypt_bytes(enc[i]) == clear[i] for i in range(nb))
    ok_pub = all(ck.decrypt_bytes(pub[i]) == clear[i] for i in range(nb))

    # the public path against the encrypted path fed trivial ciphertexts (noise level 0) of the same blocks
    triv = np.zeros((nb, 16, 8, L1), dtype=np.uint64)
    triv[..., -1] = np.unpackbits(blocks, axis=1).reshape(nb, 16, 8).astype(np.uint64) << np.uint64(63)
    triv_dev = torch.from_numpy(triv.view(np.int64)).to(device)
    ctx.aes_encrypt_blocks_dev(nb, triv_dev.data_ptr(), out_enc.data_ptr(), in_noise_sq=0)
    identical = bool(np.array_equal(out_enc.cpu().numpy().view(np.uint64), pub))
    del triv_dev

    # one host-buffer transcipher of nb·16 bytes (H2D of the plan, D2H of the output inside)
    msg = np.random.default_rng(SEED).bytes(16 * nb)
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    ct = Cipher(algorithms.AES(CLI_KEY), modes.CTR(bytes(blocks[0]))).encryptor().update(msg)
    torch.cuda.synchronize(device)
    t0 = time.perf_counter()
    tr = ctx.aes_ctr_transcipher(CLI_IV, 1, ct)
    transcipher_s = time.perf_counter() - t0
    ok_tr = ck.decrypt_bytes(tr) == msg

    info = gpu_info(args.device)
    rate = {k: nb / (np.mean(v) * 1e-3) for k, v in ms.items()}
    line = {
        "metric": "fhe_aes128_ctr_keystream_blocks_per_s", "unit": "blocks/s", "blocks": nb, "rounds": 10,
        "steps": args.steps, "warmup": args.warmup, "parameter_set": "params_sqrd_lvl_64 (n=677,k=4,N=512)",
        "encrypted": {"value": rate["encrypted"], "ms_per_step": ms["encrypted"], "boxes_per_round": [16 * nb] * 10},
        "public": {"value": rate["public"], "ms_per_step": ms["public"], "boxes_per_round": plan},
        "ratio": rate["public"] / rate["encrypted"], "box_ratio": 160 * nb / sum(plan),
        "transcipher_host": {"bytes": len(msg), "wall_s": transcipher_s, "blocks_per_s": nb / transcipher_s},
        "gpu": info, "verified": bool(ok_enc and ok_pub and ok_tr), "identical": identical,
    }
    print(json.dumps(line), flush=True)
    if not (line["verified"] and identical):
        raise SystemExit("ctr_bench: check FAILED")


if __name__ == "__main__":
    main()
