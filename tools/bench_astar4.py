#!/usr/bin/env python
"""What the astar_4 human walk costs (DESIGN 4.7), measured in one process on one GPU.

  1. generate_scenario_device with human_path="bfs" against "astar4", interleaved round by round, CUDA events, medians:
     65 536 warehouse worlds of 40x60 with 32 agents (the training env's batch), and 4 096 density worlds of 128x128.
     The outputs of the two modes are compared (everything but the walk's inner cells must be equal).
  2. scenario_from_fixed_episode_infos for 4 096 synthetic episodes, host (astar_path per leg) against device=
     (one mapf_astar4_paths call), both movement types, medians of wall time; the results must be byte-identical.

python tools/bench_astar4.py [--rounds R] [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from primal_ppo_b200 import generate_scenario_device  # noqa: E402
from primal_ppo_b200.episode_io import scenario_from_fixed_episode_infos  # noqa: E402

LINES = []


def say(s=""):
    print(s, flush=True)
    LINES.append(s)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    return q[torch.cuda.current_device()]


def gen_ms(kw, mode):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    d = generate_scenario_device(**kw, human_path=mode)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), d


def synthetic_infos(n, seed):
    """n episodes on density maps of 10..40 per side: 4 agents, 8 human poses drawn from the 4-connected component of
    the first, so that every leg has a path."""
    from collections import deque
    rng = np.random.default_rng(seed)
    infos = {k: [] for k in ("obstacleMap", "agentsSequence", "humanSequence", "humanStart", "humanGoal")}
    while len(infos["obstacleMap"]) < n:
        h, w = (int(x) for x in rng.integers(10, 41, 2))
        m = -(rng.random((h, w)) < rng.uniform(0.0, 0.3)).astype(np.int64)
        free = np.argwhere(m == 0)
        s = tuple(int(x) for x in free[rng.integers(len(free))])
        seen, q = {s}, deque([s])
        while q:
            r, c = q.popleft()
            for nb in ((r + 1, c), (r - 1, c), (r, c + 1), (r, c - 1)):
                if 0 <= nb[0] < h and 0 <= nb[1] < w and m[nb] == 0 and nb not in seen:
                    seen.add(nb)
                    q.append(nb)
        comp = sorted(seen)
        if len(comp) < 8:
            continue
        seq = [s]
        while len(seq) < 8:
            p = comp[rng.integers(len(comp))]
            if p != seq[-1]:
                seq.append(p)
        infos["obstacleMap"].append(m)
        infos["humanStart"].append(s)
        infos["humanGoal"].append(seq[1])
        infos["humanSequence"].append(seq)
        infos["agentsSequence"].append([[tuple(int(x) for x in free[rng.integers(len(free))]) for _ in range(4)] for _ in range(4)])
    infos["numEpisodes"] = n
    return infos


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    say(f"# astar_4 human walk: one {gpu_info()} (name, power limit, max SM clock), torch {torch.__version__}")
    say("## 1. generate_scenario_device, human_path bfs vs astar4 (interleaved rounds, CUDA events, median ms)")
    shapes = {"65 536 warehouse worlds 40x60, 32 agents": dict(num_worlds=65536, height=40, width=60, num_agents=32,
                                                              kind="warehouse", queue_len=16, seed=11),
              "4 096 density worlds 128x128, 32 agents": dict(num_worlds=4096, height=128, width=128, num_agents=32,
                                                              kind="density", density=(0.0, 0.3), queue_len=16, seed=12)}
    for name, kw in shapes.items():
        for mode in ("bfs", "astar4"):                   # warm-up: module load, shared-memory attribute
            gen_ms(kw, mode)
        t, same = {"bfs": [], "astar4": []}, True
        for _ in range(args.rounds):
            for mode in ("bfs", "astar4"):
                ms, d = gen_ms(kw, mode)
                t[mode].append(ms)
                out = {k: getattr(d, k) for k in ("obst", "dims", "starts", "goal_queue", "hlen", "gen_err")}
                if mode == "bfs":
                    ref = out
                else:
                    same &= all(torch.equal(out[k], ref[k]) for k in out)
                del d
        mb, ma = float(np.median(t["bfs"])), float(np.median(t["astar4"]))
        say(f"{name}: bfs {mb:.2f} ms, astar4 {ma:.2f} ms (x{ma / mb:.2f}; rounds bfs {[round(x, 2) for x in t['bfs']]}, "
            f"astar4 {[round(x, 2) for x in t['astar4']]}); maps, starts, goals, lengths, flags identical: {same}")
        torch.cuda.empty_cache()
    say("## 2. scenario_from_fixed_episode_infos, 4 096 episodes (maps 10..40, 8 human poses), host vs device (median s)")
    infos = synthetic_infos(4096, 3)
    for mtype, label in ((0, "LoopingHuman"), (1, "FixedPathHuman, max_steps 256")):
        kw = dict(human_movement_type=mtype, max_steps=256)
        scenario_from_fixed_episode_infos(infos, device="cuda:0", **{**kw, "episodes": range(8)})   # warm-up
        t, same = {"host": [], "device": []}, True
        for _ in range(3):
            for mode in ("host", "device"):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                sc = scenario_from_fixed_episode_infos(infos, device=None if mode == "host" else "cuda:0", **kw)
                torch.cuda.synchronize()
                t[mode].append(time.perf_counter() - t0)
                if mode == "host":
                    ref = sc
                else:
                    same &= all(getattr(sc, k).tobytes() == getattr(ref, k).tobytes()
                               for k in ("obst", "starts", "goal_queue", "htrace", "hlen", "hp5", "dims"))
        mh, md = float(np.median(t["host"])), float(np.median(t["device"]))
        say(f"{label}: host {mh:.3f} s, device {md:.3f} s (x{mh / md:.1f} faster); byte-identical: {same}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
