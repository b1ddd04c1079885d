#!/usr/bin/env python
"""multikey_bench.py — AES under many keys on one B200: one keyed call against a loop of single-key calls.

    python tools/multikey_bench.py [--keys 128] [--steps 2] [--warmup 1] [--device 0]

A transciphering server holds FHE(k_i) for many senders.  Each pair of arms does the same bootstraps for the same blocks;
only the batching differs (params_sqrd_lvl_64, 10-round AES-128, K = --keys distinct random keys):
  a  K blocks under K keys:  tac_aes_encrypt_blocks_keyed_dev in one call  vs  K × (tac_aes_set_key_schedule + 1-block
     tac_aes_encrypt_blocks_dev)
  b  16 keys × K/16 blocks:  one keyed call  vs  16 × (set_key_schedule + K/16-block call)
  c  AES-CTR transciphering of K one-block messages from K senders (host buffers, copies included):
     aes_ctr_transcipher_many  vs  K × (set_key_schedule + aes_ctr_transcipher)
  d  key expansion of K keys: tac_aes_key_table  vs  K sequential tac_aes_key_schedule calls (both copy their schedules
     to the host); and one key alone through tac_aes_key_schedule and through tac_aes_key_table
Timed steps alternate between all arms, each timed on the host around work that ends in a device synchronisation.  Every
arm is decrypted and compared with clear AES, and each keyed output must equal its loop's output word for word.  Prints
one JSON line with the card's name and power limit.
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

from bench import SEED, clear_aes, clear_key_schedule  # noqa: E402
from ctr_bench import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--keys", type=int, default=128, help="senders / keys K (a multiple of 16)")
    ap.add_argument("--steps", type=int, default=2, help="timed steps per arm (alternating)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args()
    if args.keys < 16 or args.keys % 16 or args.steps < 1 or args.warmup < 0:
        ap.error("--keys must be a positive multiple of 16, --steps >= 1, --warmup >= 0")

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("multikey_bench.py needs a CUDA device")
    tac = importlib.import_module("tfhe-aes-2_b200")
    device = torch.device("cuda", args.device)
    torch.cuda.set_device(device)
    stream = torch.cuda.current_stream(device)

    ck = tac.ClientKey(64, seed=SEED).gen_eval_keys()
    ctx = tac.FheContext(ck.params, device=args.device, stream=stream.cuda_stream)
    ctx.upload_keys(ck)
    K, L1 = args.keys, ck.params.big_lwe_size
    G, per = 16, args.keys // 16                     # arm b: 16 keys × per blocks
    rng = np.random.default_rng(SEED)
    keys = [rng.bytes(16) for _ in range(K)]
    blocks = [rng.bytes(16) for _ in range(K)]
    key_bits = np.stack([ck.encrypt_bytes(k, first_index=(1 << 40) + 128 * i) for i, k in enumerate(keys)])
    in_np = np.stack([ck.encrypt_bytes(b, first_index=(1 << 41) + 128 * i) for i, b in enumerate(blocks)])
    in_dev = torch.from_numpy(in_np.view(np.int64)).to(device)
    blk_bytes = 16 * 8 * L1 * 8
    kidx_a = np.arange(K, dtype=np.int32)
    kidx_b = np.repeat(np.arange(G, dtype=np.int32), per)
    ivs = [rng.bytes(8) for _ in range(K)]
    msgs = [rng.bytes(16) for _ in range(K)]
    cts = [bytes(m ^ s for m, s in zip(msgs[i], clear_aes(keys[i], ivs[i] + (1).to_bytes(8, "big")))) for i in range(K)]

    out = {name: torch.empty_like(in_dev) for name in ("a_keyed", "a_loop", "b_keyed", "b_loop")}
    res = {}
    scheds = ctx.aes_key_table(key_bits)            # the schedules the loops upload, and the table the keyed arms use

    def ptr(t, blk):
        return t.data_ptr() + blk * blk_bytes

    def a_loop():
        for k in range(K):
            ctx.aes_set_key_schedule(scheds[k])
            ctx.aes_encrypt_blocks_dev(1, ptr(in_dev, k), ptr(out["a_loop"], k))

    def b_loop():
        for g in range(G):
            ctx.aes_set_key_schedule(scheds[g])
            ctx.aes_encrypt_blocks_dev(per, ptr(in_dev, g * per), ptr(out["b_loop"], g * per))

    def c_loop():
        res["c_loop"] = []
        for i in range(K):
            ctx.aes_set_key_schedule(scheds[i])
            res["c_loop"].append(ctx.aes_ctr_transcipher(ivs[i], 1, cts[i]))

    def d_table():
        res["d_table"] = ctx.aes_key_table(key_bits)

    def d_sequential():
        res["d_sequential"] = [ctx.aes_key_schedule(key_bits[k]) for k in range(K)]

    arms = {
        # one-key expansion first: aes_key_table of one key replaces the table, d_table restores the K-key table after it
        "d_single_key_schedule": lambda: res.__setitem__("d_single", ctx.aes_key_schedule(key_bits[0])),
        "d_single_key_table": lambda: res.__setitem__("d_single_table", ctx.aes_key_table(key_bits[:1])),
        "d_table": d_table,
        "d_sequential": d_sequential,
        "a_keyed": lambda: ctx.aes_encrypt_blocks_keyed_dev(K, kidx_a, in_dev.data_ptr(), out["a_keyed"].data_ptr()),
        "a_loop": a_loop,
        "b_keyed": lambda: ctx.aes_encrypt_blocks_keyed_dev(K, kidx_b, in_dev.data_ptr(), out["b_keyed"].data_ptr()),
        "b_loop": b_loop,
        "c_keyed": lambda: res.__setitem__("c_keyed", ctx.aes_ctr_transcipher_many([(i, ivs[i], 1, cts[i]) for i in range(K)])),
        "c_loop": c_loop,
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

    # checks: clear AES for every arm, and word identity of each keyed arm with its loop
    host = {k: v.cpu().numpy().view(np.uint64) for k, v in out.items()}
    want_a = [clear_aes(keys[k], blocks[k]) for k in range(K)]
    want_b = [clear_aes(keys[kidx_b[i]], blocks[i]) for i in range(K)]
    verified = {
        "a": all(ck.decrypt_bytes(host[arm][i]) == want_a[i] for arm in ("a_keyed", "a_loop") for i in range(K)),
        "b": all(ck.decrypt_bytes(host[arm][i]) == want_b[i] for arm in ("b_keyed", "b_loop") for i in range(K)),
        "c": all(ck.decrypt_bytes(res[arm][i]) == msgs[i] for arm in ("c_keyed", "c_loop") for i in range(K)),
        "d": all(ck.decrypt_bytes(res["d_table"][k].reshape(-1, L1)) == clear_key_schedule(keys[k]) for k in range(K)),
    }
    identical = {
        "a": bool(np.array_equal(host["a_keyed"], host["a_loop"])),
        "b": bool(np.array_equal(host["b_keyed"], host["b_loop"])),
        "c": all(np.array_equal(x, y) for x, y in zip(res["c_keyed"], res["c_loop"])),
        "d": all(np.array_equal(res["d_table"][k], res["d_sequential"][k]) for k in range(K))
        and np.array_equal(res["d_single"], res["d_table"][0]) and np.array_equal(res["d_single_table"][0], res["d_table"][0]),
    }

    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    pair = lambda arm, n: {"keyed_blocks_per_s": n / (mean[arm + "_keyed"] * 1e-3), "loop_blocks_per_s": n / (mean[arm + "_loop"] * 1e-3),
                           "speedup": mean[arm + "_loop"] / mean[arm + "_keyed"]}
    line = {
        "metric": "fhe_aes128_multikey", "keys": K, "rounds": 10, "steps": args.steps, "warmup": args.warmup,
        "parameter_set": "params_sqrd_lvl_64 (n=677,k=4,N=512)",
        "a_blocks_under_distinct_keys": {"blocks": K, "keys": K, **pair("a", K)},
        "b_blocks_per_key": {"blocks": K, "keys": G, **pair("b", K)},
        "c_ctr_transcipher_senders": {"messages": K, "bytes_each": 16, **pair("c", K)},
        "d_key_expansion": {"keys": K, "table_s": mean["d_table"] * 1e-3, "sequential_s": mean["d_sequential"] * 1e-3,
                            "speedup": mean["d_sequential"] / mean["d_table"],
                            "one_key_schedule_s": mean["d_single_key_schedule"] * 1e-3, "one_key_table_s": mean["d_single_key_table"] * 1e-3},
        "ms_per_step": ms, "gpu": gpu_info(args.device), "verified": verified, "identical": identical,
    }
    print(json.dumps(line), flush=True)
    if not (all(verified.values()) and all(identical.values())):
        raise SystemExit("multikey_bench: check FAILED")


if __name__ == "__main__":
    main()
