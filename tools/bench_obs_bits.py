#!/usr/bin/env python
"""Bit-packed observations (DESIGN 4.9b): what the format buys, measured in one process on one GPU.

  1. ms per fused step (mapf_step_observe) at 65 536 x 40x40x32 and 16 384 x 80x80x128 FOV 9, f32 / bf16 / bits, the
     three formats interleaved round by round on the same env, CUDA events over >= 200 steps per format after warm-up;
     the kernel each (shape, format) launched is read from one torch.profiler pass before the timing.
  2. unpack_observations (mapf_unpack_obs): a 32 768-row random gather out of a 65 536-world bit buffer, GB/s of output.
  3. rollout buffer bytes of the observations at T = 256 (computed from shapes).
  4. one VecPPOTrainer rollout step at 1024 worlds (bf16 autocast, as bench.py's PPO extra), f32 buffer against bits.

python tools/bench_obs_bits.py [--out FILE]
"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from primal_ppo_b200 import BatchedMapfGym, random_scenario, unpack_observations  # noqa: E402
from primal_ppo_b200._cabi import obs_bits_words  # noqa: E402

LINES = []


def say(s=""):
    print(s, flush=True)
    LINES.append(s)


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[torch.cuda.current_device()] if q else "unknown"
    except (OSError, subprocess.TimeoutExpired):
        return "unknown (nvidia-smi unavailable)"


def timed(fn, n):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        fn(i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n


def kernel_names(calls):
    """The env kernels one call of each fn launches, all from ONE torch.profiler session: the calls are serialised by a
    synchronise and each launches the same number of env kernels, so the time-ordered kernel list splits evenly."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for fn in calls.values():
            torch.cuda.synchronize()
            fn(0)
            torch.cuda.synchronize()
    evs = sorted((e for e in prof.events() if e.device_type.name == "CUDA" and ("observe" in e.name or "step_kernel" in e.name)),
                 key=lambda e: e.time_range.start)
    per = max(1, len(evs) // len(calls))
    return {k: [e.name for e in evs[i * per:(i + 1) * per]] for i, k in enumerate(calls)}


def fused_setup(W, H, N, F):
    sc = random_scenario(W, H, H, N, density=(0.0, 0.3), queue_len=16, seed=100, unique_maps=256, fov=F)
    env = BatchedMapfGym(sc, use_tape=False)
    dev = env.device
    gen = torch.Generator(device=dev); gen.manual_seed(1)
    ring = [torch.randint(0, 5, (W, N), generator=gen, device=dev, dtype=torch.int8) for _ in range(8)]
    vec = torch.empty((W, N, 4), device=dev)
    bufs = {"f32": torch.empty((W, N, 6, F, F), device=dev),
            "bf16": torch.empty((W, N, 6, F, F), device=dev, dtype=torch.bfloat16),
            "bits": torch.empty(env.obs_bits_shape, device=dev, dtype=torch.int32)}
    fns = {k: (lambda i, b=b: env.step_observe(ring[i % 8], obs_out=(b, vec))) for k, b in bufs.items()}
    return env, bufs, fns


def fused_steps(shapes, rounds=8, per_round=40):
    setups = {name: fused_setup(*shape) for name, shape in shapes.items()}
    kernels = kernel_names({(name, k): fn for name, (_, _, fns) in setups.items() for k, fn in fns.items()})
    for name, (env, bufs, fns) in setups.items():
        for fn in fns.values():
            for i in range(10):
                fn(i)
        torch.cuda.synchronize()
        res = {k: [] for k in fns}
        for _ in range(rounds):
            for k, fn in fns.items():
                res[k].append(timed(fn, per_round))
        say(f"fused step, {name} ({env.W} worlds, {env.N} agents, FOV {env.F}): {rounds} interleaved rounds x {per_round} "
            f"steps per format")
        for k in fns:
            nbytes = bufs[k].numel() * bufs[k].element_size()
            say(f"  {k:4s}  median {np.median(res[k]):.4f} ms  (min {min(res[k]):.4f}, max {max(res[k]):.4f})  "
                f"observation bytes per step {nbytes / 1e6:.1f} MB")
        for k in fns:
            say(f"  {k:4s}  kernels: {'; '.join(kernels[(name, k)])}")
    del setups
    torch.cuda.empty_cache()


def unpack_rate():
    W, N, F = 65536, 32, 9
    sc = random_scenario(W, 40, 40, N, density=(0.0, 0.3), queue_len=16, seed=100, unique_maps=256)
    env = BatchedMapfGym(sc, use_tape=False)
    dev = env.device
    bits = torch.empty(env.obs_bits_shape, device=dev, dtype=torch.int32)
    env.getAllObservations(out=(bits, torch.empty((W, N, 4), device=dev)))
    gen = torch.Generator(device=dev); gen.manual_seed(2)
    rows = torch.randint(0, W, (32768,), generator=gen, device=dev)
    say(f"unpack_observations: 32768-row random gather from [{W}, {N}, {obs_bits_words(6, F)}] int32 bits")
    for dt in (torch.float32, torch.bfloat16):
        out = torch.empty((32768, N, 6, F, F), device=dev, dtype=dt)
        fn = lambda i: unpack_observations(bits, 6, F, rows=rows, dtype=dt, out=out)   # noqa: E731
        for i in range(5):
            fn(i)
        ms = [timed(fn, 20) for _ in range(5)]
        ob = out.numel() * out.element_size()
        rb = rows.numel() * (N * obs_bits_words(6, F) * 4 + 8)
        say(f"  {str(dt).split('.')[1]:8s} {np.median(ms):.4f} ms  output {ob / 1e9:.3f} GB -> {ob / np.median(ms) / 1e6:.0f} GB/s "
            f"(reads {rb / 1e6:.1f} MB)")
    del env, bits
    torch.cuda.empty_cache()


def buffer_bytes():
    T, N, C, F = 256, 32, 6, 9
    say(f"rollout buffer observations at T = {T}, 40x40x32, {C}x{F}x{F} (computed: (T+1) x W x N x bytes per agent)")
    per = {"f32": C * F * F * 4, "bf16": C * F * F * 2, "bits": obs_bits_words(C, F) * 4}
    for W in (1024, 16384, 65536):
        say(f"  W = {W:6d}: " + ", ".join(f"{k} {(T + 1) * W * N * b / 1e9:.2f} GB" for k, b in per.items()))


def trainer_step():
    from primal_ppo_b200.ppo import PPOConfig, ScrimpPolicy, VecPPOTrainer
    W, N, T = 1024, 32, 16
    sc = random_scenario(W, 40, 40, N, density=(0.0, 0.3), queue_len=16, seed=5, unique_maps=256)
    say(f"VecPPOTrainer.collect at {W} worlds x {N} agents, T = {T}, bf16 autocast: ms per rollout step "
        f"(collect time / T; includes one bootstrap forward and GAE per rollout)")
    trs = {}
    for k, od in (("f32", torch.float32), ("bits", "bits")):
        torch.manual_seed(0)
        pol = ScrimpPolicy().cuda().use_channels_last()
        trs[k] = VecPPOTrainer(BatchedMapfGym(sc, use_tape=False), pol, PPOConfig(n_steps=T), amp_dtype=torch.bfloat16,
                               obs_dtype=od)
        trs[k].collect()                      # warm-up (cuDNN algorithm choice, first launches)
    res = {k: [] for k in trs}
    for _ in range(3):
        for k, tr in trs.items():
            res[k].append(timed(lambda i: tr.collect(), 1) / T)
    for k in trs:
        say(f"  {k:4s}  median {np.median(res[k]):.3f} ms per step  ({', '.join(f'{x:.3f}' for x in res[k])})")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_obs_bits.py measures on a CUDA device; none is visible")
    say(f"GPU: {torch.cuda.get_device_name()} | nvidia-smi name, power.limit, clocks.max.sm: {gpu_info()}")
    say(f"torch {torch.__version__}, CUDA {torch.version.cuda}")
    say()
    fused_steps({"40x40x32": (65536, 40, 32, 9), "80x80x128 FOV 9": (16384, 80, 128, 9)})
    say()
    unpack_rate()
    say()
    buffer_bytes()
    say()
    trainer_step()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
