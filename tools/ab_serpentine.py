#!/usr/bin/env python
"""In-process A/B of the serpentine world order: per shape one env with ascending order forced (MAPF_DBG_FLAGS bit 12) and
one with the shipped serpentine order, same scenario, same actions, same output tensors, interleaved rounds (the mode that
runs first alternates).  Reports the median, min and max ms per call of
  - the fused step at 65 536 x 40x40x32 (f32 and bit-packed observations),
  - the two-launch step + observe at the same shape,
  - step_observe_wide at 16 384 x 80x80x128, FOV 9,
and checks that both orders reached the same state and counters.    python tools/ab_serpentine.py [rounds] [iters]"""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from primal_ppo_b200 import BatchedMapfGym, generate_scenario_device, random_scenario  # noqa: E402

ROUNDS = int(sys.argv[1]) if len(sys.argv) > 1 else 9
ITERS = int(sys.argv[2]) if len(sys.argv) > 2 else 20
MODES = {"ascending": 1 << 12, "serpentine": 0}
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(dev)} | {q}"


def make_envs(sc, **kw):
    envs = {}
    for mode, flags in MODES.items():
        os.environ["MAPF_DBG_FLAGS"] = str(flags)
        envs[mode] = BatchedMapfGym(sc, device=dev, use_tape=False, **kw)
    os.environ.pop("MAPF_DBG_FLAGS", None)
    return envs


def timed(fn):
    for i in range(3):
        fn(i)
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(ITERS):
        fn(i)
    b.record()
    torch.cuda.synchronize(dev)
    return a.elapsed_time(b) / ITERS


print("card:", card(), flush=True)
gen = torch.Generator(device=dev)
gen.manual_seed(1)

# headline shape: 65 536 worlds, 40x40, 32 agents, 6 x 9 x 9
W, N = 65536, 32
sc = random_scenario(W, 40, 40, N, density=(0.0, 0.3), queue_len=16, seed=100, unique_maps=256)
small = make_envs(sc)
e0 = small["ascending"]
obs = torch.empty((W, N, 6, 9, 9), device=dev)
vec = torch.empty((W, N, 4), device=dev)
bits = torch.empty(e0.obs_bits_shape, dtype=torch.int32, device=dev)
ring = [torch.randint(0, 5, (W, N), generator=gen, device=dev, dtype=torch.int8) for _ in range(8)]

# CTA-per-world shape: 16 384 worlds, 80x80, 128 agents, FOV 9
WW, NW = 16384, 128
dsc = generate_scenario_device(WW, 80, 80, NW, kind="density", density=(0.0, 0.3), queue_len=8, seed=909, device=dev, fov=9)
wide = make_envs(dsc)
obs_w = torch.empty((WW, NW, 6, 9, 9), device=dev)
vec_w = torch.empty((WW, NW, 4), device=dev)
ring_w = [torch.randint(0, 5, (WW, NW), generator=gen, device=dev, dtype=torch.int8) for _ in range(4)]

cases = {
    "fused f32  65536x40x40x32": (small, lambda e: lambda i: e.step_observe(ring[i % 8], obs_out=(obs, vec))),
    "fused bits 65536x40x40x32": (small, lambda e: lambda i: e.step_observe(ring[i % 8], obs_out=(bits, vec))),
    "step+observe 65536x40x40x32": (small, lambda e: lambda i: (e.step(ring[i % 8]), e.getAllObservations(out=(obs, vec)))),
    "fused wide 16384x80x80x128 F9": (wide, lambda e: lambda i: e.step_observe(ring_w[i % 4], obs_out=(obs_w, vec_w))),
}
res = {c: {m: [] for m in MODES} for c in cases}
for rnd in range(ROUNDS + 1):
    order = list(MODES) if rnd % 2 == 0 else list(MODES)[::-1]
    for c, (envs, mk) in cases.items():
        for m in order:
            t = timed(mk(envs[m]))
            if rnd:                                    # round 0 warms every shape up
                res[c][m].append(t)

print(f"{ROUNDS} rounds x {ITERS} calls, ms per call (median [min, max])")
for c in cases:
    a, s = np.array(res[c]["ascending"]), np.array(res[c]["serpentine"])
    ma, ms = np.median(a), np.median(s)
    print(f"  {c:32s} ascending {ma:.4f} [{a.min():.4f}, {a.max():.4f}]  serpentine {ms:.4f} [{s.min():.4f}, {s.max():.4f}]"
          f"  serpentine vs ascending {100 * (ms - ma) / ma:+.1f} %", flush=True)
for name, envs in (("40x40x32", small), ("80x80x128", wide)):
    s1, s2 = envs["ascending"].state(), envs["serpentine"].state()
    print(f"{name}: states equal:", all(torch.equal(s1[k], s2[k]) for k in s1),
          "counters equal:", torch.equal(envs["ascending"].counters(), envs["serpentine"].counters()), flush=True)
