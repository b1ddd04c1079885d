#!/usr/bin/env python
"""bench.py — FHE AES-128 "CTR" blocks/s (BASELINE.json metric) on N B200s of one node.

    python bench.py --gpus 1 --steps K --warmup W                      # this implementation
    torchrun --nproc-per-node N ... bench.py --gpus N --steps K ...    # one rank per GPU, weak scaling
    python bench.py --impl reference --gpus N --steps K --warmup W     # the CPU path (oracle port) on the host cores

A "step" is one pass of the hot path — `Aes128Encrypt::encrypt_block` (10 rounds = 160 circuit bootstraps per block) —
over one batch of `--blocks` counter blocks per GPU (default 128 = the per-GPU shard of BASELINE config 5, the
1024-block stream on 8 GPUs).  Keys are generated once on rank 0 and replicated by NCCL broadcast; the AES key schedule
is computed once and excluded, as in the reference (src/bin/main.rs:130-139 vs :141-159).  `value` times the path with
inputs resident in HBM, `e2e` times the same call through the host-buffer C ABI entry point (H2D and D2H inside the
timed region).  Every run decrypts its outputs and checks them against clear AES.

One JSON line is printed by rank 0.  `--dump-outputs DIR` also writes what the last timed step returned (see dump_outputs).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True                                   # the tree may be read-only: bench.py writes nothing into it

METRIC = "fhe_aes128_ctr_blocks_per_s"
SEED = 2026
STREAM_BLOCKS = 10                                               # BASELINE config 4: --number-of-outputs 10
CLI_KEY = bytes.fromhex("76b8e0ada0f13d90405d6ae55386bd28")      # BASELINE config 1/4 key and iv
CLI_IV = bytes.fromhex("bdd219b8a08ded1a")
# algorithmic f64 work (BASELINE.md §3): external product l=3 and l=1, forward FFT of one polynomial (N = 512)
F_EP3, F_EP1, F_FFT = 389120.0, 168960.0, 11776.0
FLOP_PER_PBS = 677 * F_EP3
FLOP_PER_BLOCK = 1280 * FLOP_PER_PBS + 28672 * F_EP1 + 32000 * F_FFT


def clear_aes(key, block):
    from cryptography.hazmat.primitives.ciphers import Cipher, algorithms, modes
    return Cipher(algorithms.AES(key), modes.ECB()).encryptor().update(block)


def clear_key_schedule(key):
    """AES-128 key expansion (FIPS-197 §5.2); the S-box is derived from clear AES itself so no table is duplicated here"""
    sbox = _sbox()
    rc = [0x00, 0x01, 0x02, 0x04, 0x08, 0x10, 0x20, 0x40, 0x80, 0x1B, 0x36]
    w = [list(key[4 * i:4 * i + 4]) for i in range(4)]
    for i in range(4, 44):
        t = list(w[i - 1])
        if i % 4 == 0:
            t = [sbox[t[1]] ^ rc[i // 4], sbox[t[2]], sbox[t[3]], sbox[t[0]]]
        w.append([a ^ b for a, b in zip(w[i - 4], t)])
    return bytes(b for word in w for b in word)


_SBOX = None


def _sbox():
    global _SBOX
    if _SBOX is None:
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
        _SBOX = s
    return _SBOX


def counter_blocks(first_ctr, n):
    return [CLI_IV + (first_ctr + i).to_bytes(8, "big") for i in range(n)]          # reference main.rs:108-115


DUMP_CTS = 1024                                                  # sampled output ciphertexts: 1024 x 2049 words = 16.8 MB


def dump_outputs(path, ck, out):
    """Writes what the timed path returned in its last step, so that two builds can be compared output for output (keys and
    inputs are seeded, hence identical from run to run).  Torus words are stored as signed fractions of the torus, w / 2^64.
      out_phases.npy       [blocks][16][8] float64  decrypted phase of every output bit ciphertext (secret key of the seed);
                                                    two correct builds agree on it to within the noise, whatever their f64 order
      out_ciphertexts.npy  [<=1024][2049] float64   the output LWE ciphertexts of a fixed sample of bits: rows
                                                    sorted(default_rng(SEED).choice(blocks*128, 1024, replace=False)) of the
                                                    [blocks*128][2049] output (all of it is 268 MB at 128 blocks)"""
    os.makedirs(path, exist_ok=True)
    L1 = ck.params.big_lwe_size
    flat = out.reshape(-1, L1)
    phases = ck.decrypt_phases(flat).view(np.int64).reshape(out.shape[:-1])
    rows = np.sort(np.random.default_rng(SEED).choice(flat.shape[0], min(DUMP_CTS, flat.shape[0]), replace=False))
    np.save(os.path.join(path, "out_phases.npy"), phases.astype(np.float64) * 2.0**-64)
    np.save(os.path.join(path, "out_ciphertexts.npy"), flat[rows].view(np.int64).astype(np.float64) * 2.0**-64)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)"""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.idx)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons, power = [], [], set(), []
        for r in rows:
            if len(r) < 8:
                continue
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), power_w_max=float(max(power)), samples=len(sm))
        return out


# ================================================================================================ CPU arm (oracle port)
class CpuArm:
    """The reference's CPU path for this workload: `Aes128Encrypt::encrypt_block` over whole counter blocks
    (oracle/oracle.cpp aes_encrypt_blocks = fhe_sbox_gal_mul_pbs.rs:84-132: 10 rounds, 160 circuit bootstraps and all
    leveled XORs per block), fanned out over blocks x 16 SBOX bytes on all host threads like the reference's rayon
    (main.rs:148-152, fhe_sbox_gal_mul_pbs.rs:33-41), decrypt-checked against clear AES.  The Rust reference cannot be
    built in this image, so the C++ restatement ("port") stands in; its FFT is scalar radix-2, tfhe-fft's AVX-512 plans
    would be faster (DESIGN.md section 4)."""

    def __init__(self, cores=None):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as ol          # the checker doubles as the CPU baseline: bench.py may execute oracle/ for this leg only
        self.ol = ol
        self.cores = cores or os.cpu_count() or 1
        ol.lib().orc_set_threads(self.cores)
        self.orc = ol.Oracle(64, seed=SEED)
        # one SBOX call keeps one thread busy: blocks per step = enough 16-byte states to occupy every core
        self.n_blocks = max(1, self.cores // 16)
        self.key_sched = self.orc.encrypt_bytes(clear_key_schedule(CLI_KEY), first_index=1 << 40)      # precomputed, as on the GPU arm
        self.clear = counter_blocks(1, self.n_blocks)
        self.blocks = np.stack([self.orc.encrypt_bytes(b, first_index=(1 + i) * 128) for i, b in enumerate(self.clear)])

    def step(self, rounds=10):
        """one pass over the batch; returns wall seconds (the decrypt check is outside the timed region)"""
        t0 = time.perf_counter()
        out = self.orc.aes_encrypt_blocks(self.key_sched, self.blocks, rounds=rounds)
        dt = time.perf_counter() - t0
        if rounds == 10:
            for i, blk in enumerate(self.clear):
                assert self.orc.decrypt_bytes(out[i].reshape(-1, self.orc.big1)) == clear_aes(CLI_KEY, blk), "CPU arm failed its decrypt check"
        return dt

    def describe(self, what):
        return (f"oracle C++ port (oracle/oracle.cpp aes_encrypt_blocks), {self.cores} threads, {self.n_blocks} whole block(s) per step "
                f"(10 rounds = 160 circuit bootstraps + all leveled XORs each), decrypt-verified; {what}")


def cpu_baseline_sample(budget_s=30.0):
    """bounded CPU sample for the GPU arm's line: one whole-block step if it fits the budget, else a reduced-round step scaled
    by its circuit-bootstrap count (stated in `sample`)."""
    arm = CpuArm()
    t2 = arm.step(rounds=2)                                   # 16 x (8->24) + 16 x (8->8): probe
    if t2 * 5.5 <= budget_s:
        dt = arm.step()
        return arm.n_blocks / dt, arm.cores, arm.describe(f"measured: one step = {dt:.2f} s")
    est = t2 * (9 * 1.0 + 1.0) / 2.0                          # 9 SBOX*{1,2,3} rounds + 1 SBOX round; the two kinds cost the same within 2 %
    return arm.n_blocks / est, arm.cores, arm.describe(f"a whole block exceeds the {budget_s:.0f} s budget on this host: 2-round step = {t2:.2f} s, scaled x5 (10 rounds)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm()
    for _ in range(args.warmup):
        arm.step()
    times = [arm.step() for _ in range(max(1, args.steps))]
    ms_per_step = 1e3 * float(np.mean(times))
    value = arm.n_blocks / (ms_per_step * 1e-3)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "blocks/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": "blocks/s", "cores": arm.cores, "kind": "port",
                         "sample": arm.describe(f"every step measured (min {min(times):.2f} s, max {max(times):.2f} s)"), "blocks_per_step": arm.n_blocks},
        "e2e": {"value": value, "unit": "blocks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "verified": True,
    }
    print(json.dumps(line), flush=True)


PBS_SOURCES = ("tac_common.h", "ep_core.cuh", "ep_step.cuh", "kernels_ep.cuh", "kernels_shape.inl", "kernels_n512.cu", "shape_launch.h")


def csrc_digest():
    """sha256 over the sources the PBS kernels are compiled from: ties a committed ncu capture to the code it profiled (the GPU box
    has no .git, so a commit hash cannot be checked there)"""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "tfhe-aes-2_b200", "csrc")
    for name in PBS_SOURCES:
        h.update(name.encode() + b"\0" + open(os.path.join(d, name), "rb").read())
    return h.hexdigest()[:16]


def pbs_traffic(n_ct):
    """dram__bytes_read.sum + dram__bytes_write.sum of one PBS launch (`pbs_merged_kernel`) from the committed `ncu --set full` capture
    (profiles/pbs_dram_traffic.json), but only when that capture profiled exactly the kernel sources of this tree; otherwise None."""
    try:
        table = json.load(open(os.path.join(ROOT, "profiles", "pbs_dram_traffic.json")))
        if table.get("csrc_sha16") != csrc_digest():
            return None
        return table.get("bytes_per_launch", {}).get(str(n_ct))
    except Exception:
        return None


def tensor_roofline(n_ct, pfks_ms):
    ops = 2.0 * 15 * 4098 * 12800 * n_ct
    achieved = ops / (pfks_ms * 1e-3) / 1e12 if pfks_ms > 0 else None
    peak, src = 4500.0, "nominal dense int8 (MEASURED_PEAKS.json absent)"
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, src = 2.0 * float(mp["bf16_tflops"]), "2 x measured dense bf16 (MEASURED_PEAKS.json bf16_tflops)"
    except Exception:
        pass
    return {"bound": "tensor", "kernel": "umma_digit_tiles_kernel + lwe_gemm_umma_kernel<2> + pfks_fixup_kernel", "achieved": achieved, "peak": peak, "unit": "TOP/s (u8)",
            "frac": achieved / peak if achieved else None, "peak_source": src, "avg_stage_ms": pfks_ms}


def workload_config(args):
    """identical for both arms (the CPU arm processes the same stream a bounded number of whole blocks at a time)"""
    return {"workload": f"AES-128 CTR stream, {args.blocks} counter blocks per GPU x 10 rounds (per-GPU shard of BASELINE config 5: 1024 blocks / 8 GPUs), "
                        "params_sqrd_lvl_64, key schedule precomputed", "blocks_per_gpu": args.blocks, "rounds": 10,
            "parameter_set": "params_sqrd_lvl_64 (n=677,k=4,N=512)", "sharding": "contiguous counter ranges per GPU, no per-round collective",
            "l2": "inputs larger than L2: 672 MB of keys + >= 268 MB of state are streamed every round"}


# ================================================================================================ GPU arm
def run_gpu(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run --nproc-per-node N")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout for the one JSON line
        dist.init_process_group("nccl", device_id=device)
    tac = importlib.import_module("tfhe-aes-2_b200")
    dmod = importlib.import_module("tfhe-aes-2_b200.distributed")

    stream = torch.cuda.current_stream(device)
    t_setup = time.perf_counter()
    ck = tac.ClientKey(64, seed=SEED)                      # every rank derives the same secret keys from the seed (client side)
    ctx = tac.FheContext(ck.params, device=local_rank, stream=stream.cuda_stream)
    key_sched_host = None
    if rank == 0:
        ck.gen_eval_keys()
        key_sched_host = ck.encrypt_bytes(clear_key_schedule(CLI_KEY), first_index=1 << 40)
    if world > 1:
        key_bytes = dmod.replicate_keys(ctx, ck if rank == 0 else None, device)
        key_bytes += dmod.replicate_key_schedule(ctx, key_sched_host, device)
    else:
        ctx.upload_keys(ck)
        ctx.aes_set_key_schedule(key_sched_host)
        key_bytes = 0
    L1 = ck.params.big_lwe_size
    nb = args.blocks
    first_ctr = 1 + rank * nb
    blocks_clear = counter_blocks(first_ctr, nb)
    in_host = torch.empty((nb, 16, 8, L1), dtype=torch.int64).pin_memory()
    out_host = torch.empty_like(in_host).pin_memory()
    in_np = in_host.numpy().view(np.uint64)
    for i, blk in enumerate(blocks_clear):
        in_np[i] = ck.encrypt_bytes(blk, first_index=(first_ctr + i) * 128)
    in_dev = in_host.to(device, non_blocking=False)
    out_dev = torch.empty_like(in_dev)
    torch.cuda.synchronize(device)
    setup_s = time.perf_counter() - t_setup

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    def step_dev():
        ctx.aes_encrypt_blocks_dev(nb, in_dev.data_ptr(), out_dev.data_ptr(), rounds=10)

    def step_e2e():
        rc = ctx.L.tac_aes_encrypt_blocks(ctx.h, nb, 10, 1, in_host.data_ptr(), out_host.data_ptr())
        ctx._check(rc)

    fp64_peak = ctx.fp64_peak_tflops()

    # ---- device-resident timing
    for _ in range(args.warmup):
        step_dev()
    barrier()
    ctx.stage_times()                      # reset
    ctx.set_profiling(True)                # CUDA events around every stage, no host sync
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ctx.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_dev()
    e1.record(stream)
    barrier()
    ms_total = e0.elapsed_time(e1)
    launches = ctx.launch_count() - launches0
    stages = ctx.stage_times()
    ctx.set_profiling(False)
    clocks = sampler.stop()
    # decrypt-verify this rank's outputs against clear AES (every block)
    got = out_dev.cpu().numpy().view(np.uint64)
    ok = all(ck.decrypt_bytes(got[i]) == clear_aes(CLI_KEY, blocks_clear[i]) for i in range(nb))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ck, got)

    # ---- end-to-end timing through the host-buffer entry point (pinned host memory, H2D + D2H inside)
    e2e_steps = max(1, args.steps)
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    ok_e2e = all(ck.decrypt_bytes(out_host.numpy().view(np.uint64)[i]) == clear_aes(CLI_KEY, blocks_clear[i]) for i in (0, nb - 1))

    # ---- per-block latency: one block alone (128 ciphertexts in flight)
    lat_ms = None
    if rank == 0:
        one_in, one_out = in_dev[:1].contiguous(), torch.empty_like(in_dev[:1])
        ctx.aes_encrypt_blocks_dev(1, one_in.data_ptr(), one_out.data_ptr(), rounds=10)
        torch.cuda.synchronize(device)
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0.record(stream)
        ctx.aes_encrypt_blocks_dev(1, one_in.data_ptr(), one_out.data_ptr(), rounds=10)
        l1.record(stream)
        torch.cuda.synchronize(device)
        lat_ms = l0.elapsed_time(l1)

    # ---- BASELINE config 4: the reference's default scenario, a 10-block stream (main.rs --number-of-outputs 10), split over
    # the ranks by contiguous counter ranges (strong scaling), through the host-buffer entry point (H2D + D2H inside)
    s0, s1 = dmod.shard_range(STREAM_BLOCKS, rank, world)
    n_mine = s1 - s0
    st_in = torch.empty((max(1, n_mine), 16, 8, L1), dtype=torch.int64).pin_memory()
    st_out = torch.empty_like(st_in).pin_memory()
    st_clear = counter_blocks(1 + s0, n_mine)
    for i, blk in enumerate(st_clear):
        st_in.numpy().view(np.uint64)[i] = ck.encrypt_bytes(blk, first_index=(1 << 41) + (s0 + i) * 128)

    def stream_pass():
        if n_mine:
            ctx._check(ctx.L.tac_aes_encrypt_blocks(ctx.h, n_mine, 10, 1, st_in.data_ptr(), st_out.data_ptr()))

    stream_pass()
    stream_s = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        stream_pass()
        barrier()
        stream_s.append(time.perf_counter() - t0)
    ok_stream = all(ck.decrypt_bytes(st_out.numpy().view(np.uint64)[i]) == clear_aes(CLI_KEY, st_clear[i]) for i in range(n_mine))

    # ---- key expansion on the device (the reference prints it separately: main.rs:130-139); rank 0 only
    key_exp_s, ok_ks = None, True
    if rank == 0 and not args.no_key_expansion:
        key_bits = ck.encrypt_bytes(CLI_KEY, first_index=1 << 42)
        ctx.aes_key_schedule(key_bits)                                  # warm-up (LUT registration, workspaces)
        t0 = time.perf_counter()
        ks_fhe = ctx.aes_key_schedule(key_bits)
        key_exp_s = time.perf_counter() - t0
        ok_ks = ck.decrypt_bytes(ks_fhe.reshape(-1, L1)) == clear_key_schedule(CLI_KEY)

    # ---- reduce over ranks: max time, sum of launches, all verified
    ok_local = ok and ok_e2e and ok_stream and ok_ks
    red = torch.tensor([ms_total, e2e_s, float(launches), 1.0 if ok_local else 0.0, float(np.mean(stream_s))], dtype=torch.float64, device=device)
    if world > 1:
        mx = red.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = red.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        mn = red.clone(); dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        ms_total, e2e_s, launches, ok_all, stream_wall = float(mx[0]), float(mx[1]), int(sm[2]), bool(mn[3] > 0.5), float(mx[4])
    else:
        ok_all, stream_wall = ok_local, float(np.mean(stream_s))

    if rank == 0:
        total_blocks = nb * world
        ms_per_step = ms_total / args.steps
        value = total_blocks / (ms_per_step * 1e-3)
        e2e_value = total_blocks * e2e_steps / e2e_s
        pbs_launches = max(1, stages["passes"])
        pbs_ms = stages["pbs"] / pbs_launches
        n_ct_per_launch = nb * 128 / max(1, (pbs_launches // (10 * args.steps)))
        achieved = n_ct_per_launch * FLOP_PER_PBS / (pbs_ms * 1e-3) / 1e12
        stage_share = {k: round(v / max(1e-9, sum(stages[s] for s in ("keyswitch", "pbs", "pfks", "ggsw_fft", "vertical_packing"))), 4)
                       for k, v in stages.items() if k != "passes"}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            v, cores, desc = cpu_baseline_sample(budget_s=30.0)
            cpu = {"value": v, "unit": "blocks/s", "cores": cores, "kind": "port", "sample": desc}
        line = {
            "metric": METRIC, "value": value, "unit": "blocks/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "blocks/s", "h2d_bytes_per_step": int(in_host.numel() * 8 * world),
                    "d2h_bytes_per_step": int(out_host.numel() * 8 * world), "steps": e2e_steps},
            "gpu_launches": int(launches),
            "roofline": {"bound": "fp64", "kernel": "pbs_merged_kernel<N=512,k=4,l=3,B=3,256 threads>", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": achieved / fp64_peak if fp64_peak else None, "traffic": pbs_traffic(int(n_ct_per_launch)),
                         "peak_source": "DFMA microbenchmark in this run (FP64 is not in MEASURED_PEAKS.json)",
                         "peak_nominal": 37.2, "frac_of_nominal": achieved / 37.2, "peak_nominal_source": "148 SM x 64 DFMA/clk x 2 flop x 1.965 GHz",
                         "algorithmic_flop_per_launch": n_ct_per_launch * FLOP_PER_PBS, "avg_launch_ms": pbs_ms, "launches": int(pbs_launches),
                         "whole_step_frac": value / world * FLOP_PER_BLOCK / 1e12 / fp64_peak if fp64_peak else None},
            # secondary: the PFKS stage (digit tiles + tcgen05 kind::i8 GEMM + fix-up) against the tensor roofline.  Algorithmic
            # work: 787 M u8 multiply-accumulates per ciphertext (15 byte-limb products × 4098 digits × 12800 columns); peak: twice the
            # measured dense bf16 throughput of MEASURED_PEAKS.json (int8 runs at 2× bf16 on the B200 tensor cores; nominal 4500 TOP/s).
            "roofline_tensor": tensor_roofline(n_ct_per_launch, stages["pfks"] / pbs_launches),
            "stage_share": stage_share,
            "cpu_baseline": cpu,
            "latency_s_per_block": None if lat_ms is None else lat_ms * 1e-3,
            # BASELINE config 4 (10-block stream, strong scaling over the ranks): wall time until all ten blocks are back on the
            # host, through tac_aes_encrypt_blocks with host buffers; mean of 3 passes, max over ranks
            "stream10": {"blocks": STREAM_BLOCKS, "n_gpus": world, "split": [dmod.shard_range(STREAM_BLOCKS, r, world)[1] - dmod.shard_range(STREAM_BLOCKS, r, world)[0] for r in range(world)],
                         "wall_s": stream_wall, "blocks_per_s": STREAM_BLOCKS / stream_wall, "scaling": "strong"},
            "key_expansion_s": key_exp_s,
            "verified": ok_all, "setup_s": setup_s, "key_broadcast_bytes": int(key_bytes),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not ok_all:
        raise SystemExit("decrypt check against clear AES FAILED")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--blocks", type=int, default=int(os.environ.get("TAC_BENCH_BLOCKS", "128")), help="AES blocks per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-key-expansion", action="store_true", help="skip the FHE key-schedule timer")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step (rank 0's blocks) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to the GPU arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
