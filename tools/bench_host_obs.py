#!/usr/bin/env python
"""The split-phase host call with bit-packed observations and with observations in the result slot (DESIGN 4.10),
measured in one process per GPU.

  1. bench.py's end-to-end loop (run_e2e: 8 pinned action buffers, compact result slots, host_wait(1) one step behind,
     a host clock that ends in a synchronise) at 65 536 x 40x40x32, built like bench.build_scenario, with obs_dev in f32
     against bits, interleaved round by round on the same env.  The device-resident fused step (mapf_step_observe, CUDA
     events) of both formats is timed in the same rounds for reference.
  2. MAPF_HOST_OBS with bits (compact slots, the observation block and vec copied to the host every step): ms per step and
     D2H bytes per step at W = 4096 and 65 536, with obs_dev alternating between two buffers (a rollout buffer's pattern:
     no step waits for a copy) and with one reused obs_dev (every step waits for the previous step's copy).
Under torchrun every rank runs the same loops on its own GPU behind a barrier; a figure is the slowest rank's time.

python tools/bench_host_obs.py [--rounds R] [--steps K] [--out FILE]
torchrun --nproc_per_node 8 tools/bench_host_obs.py --gpus 8 [--out FILE]
"""
import argparse
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import bench  # noqa: E402
from bench_obs_bits import gpu_info  # noqa: E402
from primal_ppo_b200 import BatchedMapfGym  # noqa: E402
from primal_ppo_b200.build import build  # noqa: E402

LINES = []
RANK, WORLD = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def say(s=""):
    if RANK == 0:
        print(s, flush=True)
        LINES.append(s)


def sync_all(dev):
    torch.cuda.synchronize(dev)
    if WORLD > 1:
        dist.barrier()


def slowest(x, dev):
    """The largest value of x over the ranks."""
    if WORLD == 1:
        return x
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def read_reward(slot):
    """The host reads a result of the step (as bench.py does): agent (0, 0)'s reward from the packed record."""
    p = int(slot["packed"][0, 0]) & 0xffff
    return (-2.0, -2.0, -2.0, -0.35, -0.3)[min(p & 7, 4)] + (1.5 if p & 8 else 0.0)


def e2e(env, ring_h, obs, vec, n_calls, dev):
    """bench.py's run_e2e with obs_dev / vec_dev taken round-robin from the lists `obs` / `vec`: ms per step of the slowest
    rank and the bytes of one step's copies (h2d, d2h)."""
    acts, slots, nb = ring_h["action_ring"], ring_h["slots"], len(obs)
    for i in range(3):
        env.step_observe_host_begin(acts[i % 8], slots[i & 1], obs[i % nb], vec[i % nb])
    env.host_wait(0)
    sync_all(dev)
    t0 = time.perf_counter()
    sink = 0.0
    for i in range(n_calls):
        h2d, d2h = env.step_observe_host_begin(acts[i % 8], slots[(i + 3) & 1], obs[i % nb], vec[i % nb])
        if i > 0:
            env.host_wait(1)                          # step i-1 has landed while step i runs
            sink += read_reward(slots[(i + 2) & 1])
    env.host_wait(0)
    sink += read_reward(slots[(n_calls + 2) & 1])
    torch.cuda.synchronize(dev)
    ms = (time.perf_counter() - t0) / n_calls * 1e3
    return slowest(ms, dev), h2d, d2h


def device_step(env, ring, obs, vec, n_calls, dev):
    """The device-resident fused step (actions already in HBM), CUDA events: ms per step of the slowest rank."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync_all(dev)
    a.record()
    for i in range(n_calls):
        env.step_observe(ring[i % 8], obs_out=(obs, vec))
    b.record()
    torch.cuda.synchronize(dev)
    return slowest(a.elapsed_time(b) / n_calls, dev)


def stats(xs):
    return f"median {np.median(xs):.4f} ms  (min {min(xs):.4f}, max {max(xs):.4f})"


def make_env(W, dev):
    sc, ring = bench.bench_inputs(W, dev, RANK)
    env = BatchedMapfGym(sc, device=dev, seed=1234 + RANK, use_tape=False)
    return env, ring


def pinned_ring(env, ring, **kw):
    h = env.make_host_ring(slots=2, action_slots=8, compact=True, **kw)
    for k, r in enumerate(ring):
        h["action_ring"][k].copy_(r)
    return h


def format_ab(dev, rounds, steps):
    W, N = 65536, bench.N_AGENTS
    env, ring = make_env(W, dev)
    vec = torch.empty((W, N, 4), device=dev)
    bufs = {"f32": torch.empty((W, N, bench.CH, bench.FOV, bench.FOV), device=dev),
            "bits": torch.empty(env.obs_bits_shape, dtype=torch.int32, device=dev)}
    ring_h = pinned_ring(env, ring)
    for k, b in bufs.items():                          # warm-up of every shape the timed loops use
        env.getAllObservations(out=(b, vec))
        e2e(env, ring_h, [b], [vec], 20, dev)
        device_step(env, ring, b, vec, 20, dev)
    res = {(k, m): [] for k in bufs for m in ("e2e", "device")}
    for _ in range(rounds):
        for k, b in bufs.items():
            res[(k, "e2e")].append(e2e(env, ring_h, [b], [vec], steps, dev)[0])
            res[(k, "device")].append(device_step(env, ring, b, vec, steps, dev))
    _, h2d, d2h = e2e(env, ring_h, [bufs["bits"]], [vec], 3, dev)
    say(f"1. split-phase loop of bench.py (compact slots, 8 pinned action buffers), {W} worlds x {N} agents, 40x40, "
        f"FOV {bench.FOV}, {WORLD} GPU(s): {rounds} interleaved rounds x {steps} steps per arm; ms per step of the slowest rank")
    for k in bufs:
        nb = bufs[k].numel() * bufs[k].element_size()
        say(f"  obs_dev {k:4s}  split-phase host call {stats(res[(k, 'e2e')])}")
        say(f"  obs_dev {k:4s}  device-resident step  {stats(res[(k, 'device')])}   (observation bytes written {nb / 1e6:.1f} MB)")
    for k in bufs:
        med = np.median(res[(k, "e2e")])
        say(f"  obs_dev {k:4s}  e2e {W * N * WORLD / med / 1e6:.1f} G agent-steps/s over {WORLD} GPU(s); per GPU per step "
            f"H2D {h2d / 1e6:.2f} MB + D2H {d2h / 1e6:.2f} MB -> {(h2d + d2h) * WORLD / med / 1e6:.1f} GB/s through the host in all")
    return env, ring


def host_obs(dev, rounds, steps, big):
    say(f"2. MAPF_HOST_OBS, bit-packed observations, compact slots: the step's bits and vec come back in the result slot; "
        f"{rounds} rounds, ms per step of the slowest rank, {WORLD} GPU(s)")
    for W in (4096, 65536):
        N = bench.N_AGENTS
        env, ring = big if W == 65536 else make_env(W, dev)
        obs = [torch.empty(env.obs_bits_shape, dtype=torch.int32, device=dev) for _ in range(2)]
        vec = [torch.empty((W, N, 4), device=dev) for _ in range(2)]
        ring_h = pinned_ring(env, ring, obs="bits")
        n = steps if W == 4096 else max(20, steps // 4)
        arms = {"two obs_dev buffers, alternating": (obs, vec), "one obs_dev buffer, reused": (obs[:1], vec[:1])}
        for o, v in arms.values():
            e2e(env, ring_h, o, v, 10, dev)
        res = {k: [] for k in arms}
        for _ in range(rounds):
            for k, (o, v) in arms.items():
                res[k].append(e2e(env, ring_h, o, v, n, dev)[0])
        _, h2d, d2h = e2e(env, ring_h, obs, vec, 3, dev)
        for k in arms:
            med = np.median(res[k])
            say(f"  W = {W:6d}, {k:34s} {stats(res[k])}  D2H {d2h / 1e6:.2f} MB/step per GPU -> "
                f"{d2h * WORLD / med / 1e6:.1f} GB/s in all")
        del env, ring, obs, vec, ring_h
        torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1, help="GPUs of the job (run under torchrun when > 1)")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_host_obs.py measures on a CUDA device; none is visible")
    if args.gpus != WORLD:
        raise SystemExit(f"--gpus {args.gpus} needs torchrun --nproc_per_node {args.gpus} (WORLD_SIZE is {WORLD})")
    build()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if WORLD > 1:
        dist.init_process_group("nccl", device_id=dev)
    say(f"GPU: {torch.cuda.get_device_name(dev)} | nvidia-smi name, power.limit, clocks.max.sm: {gpu_info()}")
    say(f"torch {torch.__version__}, CUDA {torch.version.cuda}, {WORLD} GPU(s)")
    say()
    big = format_ab(dev, args.rounds, args.steps)
    say()
    host_obs(dev, max(3, args.rounds // 2), args.steps, big)
    if args.out and RANK == 0:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")
    if WORLD > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
