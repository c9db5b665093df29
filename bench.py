#!/usr/bin/env python
"""bench.py — agent-steps/s of the MAPF hot path (step + observe) on B200, next to the CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one joint step + one observation build over all worlds of the rank (mapf_step_observe, one launch):
the rollout loop's per-step env work (runner.py:64-100) with the policy excluded (SURVEY.md §8d).
Workload (N=1) = BASELINE.json configs[2]: 65 536 lockstep 40x40 worlds, 32 agents, obstacle density U[0,0.3],
uniform random actions.  Weak scaling: every rank owns 65 536 worlds; worlds never communicate.

Printed JSON (rank 0): value = whole-job agent-steps/s with inputs resident in HBM; `e2e` = the same through the
split-phase host-buffer C-ABI call (mapf_step_observe_host_begin/_wait: every step's joint action comes from pinned host
memory and every step's per-agent results are copied back and read on the host, one step behind the launch);
`sustained` = the same device-resident loop held for >= 2 s;  `strong` / `fov_sweep` / `ppo` = BASELINE configs[2] with the
65 536 worlds split over the ranks, configs[4] and configs[3] (all ranks take part, times are max over ranks);
`roofline` for the dominant kernel (the fused step_observe_kernel) from CUDA events inside the timed region; `cpu_baseline` = the C port
of the reference's algorithm (oracle/) on this box's host cores.  `--impl reference` times that CPU path alone.
`--dump-outputs DIR` writes what the last timed step returned (rank 0) to DIR/<name>.npy, see dump_outputs().
BENCH_E2E_DEBUG=1 prints the wall time of every e2e call on stderr.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "65536 batched 40x40 worlds, 32 agents, density 0-0.3, step+observe (BASELINE.json configs[2])"
H = WD = 40
N_AGENTS = 32
FOV, CH = 9, 6


def bench_config(worlds_per_gpu):
    """The `config` object of BOTH arms (the GPU arm and `--impl reference`): the workload BASELINE.json's metric is quoted on."""
    return {"workload": WORKLOAD, "worlds_per_gpu": worlds_per_gpu, "agents": N_AGENTS, "grid": [H, WD], "fov": FOV, "channels": CH}


def algorithmic_bytes(n_agents=N_AGENTS, h=H, wd=WD, c=CH, f=FOV):
    """SURVEY.md §8d, per agent-step: step ~ 46 + (H*Wd+8)/N, observe ~ 16 + 4*C*F^2 + (H*Wd+8)/N + 8, and for the
    fused step+observe launch B = 62 + 4*C*F^2 + (H*Wd+8)/N (the world's map and human are read once)."""
    shared = (h * wd + 8) / n_agents
    step = 46 + shared
    observe = 16 + 4 * c * f * f + shared + 8
    fused = 62 + 4 * c * f * f + shared
    return step, observe, fused


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` on this workload, from the committed
    `ncu --set full` capture (profiles/traffic.json, written by tools/ncu_traffic.py); None if not captured."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        d = json.load(open(p))
        return float(d[kernel]["dram_bytes_per_launch"])
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.  NVML in-process (nvidia_ml_py) every 2 ms from a
    background thread; falls back to an `nvidia-smi -lms` child when NVML is unavailable.  Start it before the warm-up
    (`start()`), bracket the timed region with `mark_begin()` / `mark_end()`; `summary()` uses the samples in between."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thread = index, [], None, None
        self.stop = threading.Event()
        self.t0 = self.t1 = None
        self.source = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = self.index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                ent = vis.split(",")[idx].strip()
                idx = int(ent) if ent.isdigit() else idx
            h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            R = pynvml
            bits = (("hw_slowdown", getattr(R, "nvmlClocksEventReasonHwSlowdown", 0x8)),
                    ("hw_thermal_slowdown", getattr(R, "nvmlClocksEventReasonHwThermalSlowdown", 0x40)),
                    ("sw_thermal_slowdown", getattr(R, "nvmlClocksEventReasonSwThermalSlowdown", 0x20)),
                    ("sw_power_cap", getattr(R, "nvmlClocksEventReasonSwPowerCap", 0x4)))
            get_reasons = getattr(R, "nvmlDeviceGetCurrentClocksEventReasons", None) or R.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self.stop.is_set():
                    try:
                        sm = float(R.nvmlDeviceGetClockInfo(h, R.NVML_CLOCK_SM))
                        rs = int(get_reasons(h))
                        self.rows.append((time.perf_counter(), sm, mx, [n for n, b in bits if rs & b]))
                    except Exception:
                        pass
                    time.sleep(0.002)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.source = "nvml"
        except Exception:
            try:
                self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                              "--format=csv,noheader,nounits", "-lms", "20"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.thread = threading.Thread(target=self._read_smi, daemon=True)
                self.thread.start()
                self.source = "nvidia-smi"
            except Exception:
                self.proc = None
        return self

    def _read_smi(self):
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                reasons = [n for n, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6])
                           if val.lower().startswith("active")]
                self.rows.append((time.perf_counter(), float(r[0]), float(r[1]), reasons))
            except Exception:
                continue

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def close(self):
        self.stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass

    # context-manager form: the whole `with` body is the timed region
    def __enter__(self):
        if self.thread is None:
            self.start()
        self.mark_begin()
        return self

    def __exit__(self, *a):
        self.mark_end()
        time.sleep(0.01)
        self.close()

    def summary(self):
        rows = self.rows
        inside = [r for r in rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or r[0])]
        if not inside and rows and self.t0 is not None:       # region shorter than the sampling period: nearest samples
            mid = 0.5 * (self.t0 + (self.t1 or self.t0))
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:3]
        if not inside:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "source": self.source}
        reasons = sorted({n for r in inside for n in r[3]})
        return {"sm_mhz": float(np.median([r[1] for r in inside])), "sm_max_mhz": float(max(r[2] for r in inside)),
                "reasons": reasons, "samples": len(inside), "source": self.source}


def build_scenario(worlds, seed):
    from primal_ppo_b200 import random_scenario
    return random_scenario(worlds, H, WD, N_AGENTS, density=(0.0, 0.3), queue_len=16, seed=seed,
                           unique_maps=min(256, worlds), fov=FOV, num_channel=CH)


def bench_inputs(worlds, dev, rank):
    """The headline loop's inputs: the worlds and a device-resident ring of 8 joint actions, seeded from the rank only."""
    import torch
    sc = build_scenario(worlds, seed=100 + rank)
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    ring = [torch.randint(0, 5, (worlds, N_AGENTS), generator=gen, device=dev, dtype=torch.int8) for _ in range(8)]
    return sc, ring


DUMP_WORLDS = 512         # 512 worlds x ~64 KB of outputs = 33 MB on disk


def dump_outputs(out_dir, res):
    """Writes what one `env.step_observe` returned -- the StepOut fields, obs and vec -- as float32 .npy files (float64
    for int32 fields), restricted to a fixed sample of DUMP_WORLDS worlds drawn with seed 0 and kept in world order.  The
    bench's inputs depend only on its arguments, so two builds run with the same arguments can be compared file by file."""
    import torch
    out, obs, vec = res
    W = obs.shape[0]
    idx = np.sort(np.random.default_rng(0).choice(W, size=min(W, DUMP_WORLDS), replace=False))
    idx_t = torch.from_numpy(idx).to(obs.device)
    arrays = {f: getattr(out, f) for f in ("status", "reward", "cost", "train_valid", "goals_reached", "violated",
                                           "shadow_goals", "fixed_actions")}
    arrays.update(obs=obs, vec=vec)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.index_select(0, idx_t).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype == np.int32 else np.float32))


def _max_over_ranks(x, dev, world_size):
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed_env_loop(env, ring, obs, vec, steps, dev, world_size, warmup=3):
    """`steps` fused env steps, CUDA events on the launching stream, barrier + synchronize on both sides; returns
    milliseconds (max over ranks)."""
    import torch
    import torch.distributed as dist
    for i in range(warmup):
        env.step_observe(ring[i % len(ring)], obs_out=(obs, vec))
    if world_size > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        env.step_observe(ring[i % len(ring)], obs_out=(obs, vec))
    b.record()
    if world_size > 1:
        dist.barrier()
    torch.cuda.synchronize(dev)
    return _max_over_ranks(a.elapsed_time(b), dev, world_size)


def bench_strong(sc, dev, rank, world_size, steps):
    """BASELINE configs[2] as STRONG scaling (SURVEY §8): 65 536 worlds in total, 65 536 / G per GPU."""
    import torch
    from primal_ppo_b200 import BatchedMapfGym
    total = 65536
    Wl = total // world_size
    env = BatchedMapfGym(sc.slice(0, Wl), device=dev, seed=1234, use_tape=False, world_offset=rank * Wl)
    obs = torch.empty((Wl, N_AGENTS, CH, FOV, FOV), dtype=torch.float32, device=dev)
    vec = torch.empty((Wl, N_AGENTS, 4), dtype=torch.float32, device=dev)
    gen = torch.Generator(device=dev); gen.manual_seed(77 + rank)
    ring = [torch.randint(0, 5, (Wl, N_AGENTS), generator=gen, device=dev, dtype=torch.int8) for _ in range(8)]
    ms = timed_env_loop(env, ring, obs, vec, steps, dev, world_size, warmup=5)
    # the same through the split-phase host call (pinned actions in, per-agent results out, read one step behind)
    hr = env.make_host_ring(slots=2, action_slots=8, compact=True)
    for k, r in enumerate(ring):
        hr["action_ring"][k].copy_(r)
    for i in range(3):
        env.step_observe_host_begin(hr["action_ring"][i % 8], hr["slots"][i & 1], obs, vec)
    env.host_wait(0)
    if world_size > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    for i in range(steps):
        env.step_observe_host_begin(hr["action_ring"][i % 8], hr["slots"][(i + 3) & 1], obs, vec)
        if i > 0:
            env.host_wait(1)
            _ = int(hr["slots"][(i + 2) & 1]["packed"][0, 0])
    env.host_wait(0)
    torch.cuda.synchronize(dev)
    e2e_s = _max_over_ranks(time.perf_counter() - t0, dev, world_size)
    out = {"total_worlds": total, "worlds_per_gpu": Wl, "steps": steps, "ms_per_step": ms / steps,
           "value": total * N_AGENTS * steps / (ms * 1e-3), "e2e_value": total * N_AGENTS * steps / e2e_s,
           "unit": "agent-steps/s", "scaling": "strong"}
    del env, obs, vec, ring, hr
    torch.cuda.empty_cache()
    return out


FOV_SWEEP = ((9, 16384), (15, 8192), (21, 4096), (31, 2048))      # (FOV, worlds per GPU): obs <= ~6 GB per GPU


def bench_fov_sweep(dev, rank, world_size, steps=10):
    """BASELINE configs[4]: 80x80 worlds, 128 agents, FOV 9/15/21/31 (memory-bound roofline stress), worlds generated on
    the device.  Per FOV: ms per step of mapf_step_observe (max over ranks), algorithmic GB/s and fraction of the peak."""
    import torch
    from primal_ppo_b200 import BatchedMapfGym, generate_scenario_device
    H, N, C = 80, 128, 6
    peak, _ = measured_peaks()
    rows = []
    for F, W in FOV_SWEEP:
        dsc = generate_scenario_device(W, H, H, N, kind="density", density=(0.0, 0.3), queue_len=8, seed=900 + F,
                                       world_offset=rank * W, device=dev, fov=F)
        env = BatchedMapfGym(dsc, device=dev, use_tape=False, world_offset=rank * W)
        obs = torch.empty((W, N, C, F, F), device=dev); vec = torch.empty((W, N, 4), device=dev)
        gen = torch.Generator(device=dev); gen.manual_seed(F + rank)
        ring = [torch.randint(0, 5, (W, N), generator=gen, device=dev, dtype=torch.int8) for _ in range(4)]
        ms = timed_env_loop(env, ring, obs, vec, steps, dev, world_size) / steps
        # the two launches separately (local timing)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        env.step(ring[0]); env.getAllObservations(out=(obs, vec)); torch.cuda.synchronize(dev)
        ev[0].record(); env.step(ring[1]); ev[1].record(); env.getAllObservations(out=(obs, vec)); ev[2].record()
        torch.cuda.synchronize(dev)
        _, b_obs, b_all = algorithmic_bytes(N, H, H, C, F)
        rows.append({"fov": F, "worlds_per_gpu": W, "ms_per_step": ms, "agent_steps_per_s": W * N * world_size / (ms * 1e-3),
                     "step_observe_gbs": b_all * W * N / (ms * 1e-3) / 1e9, "step_observe_frac": b_all * W * N / (ms * 1e-3) / 1e9 / peak,
                     "step_ms": ev[0].elapsed_time(ev[1]), "observe_ms": ev[1].elapsed_time(ev[2]),
                     "observe_frac": b_obs * W * N / (ev[1].elapsed_time(ev[2]) * 1e-3) / 1e9 / peak,
                     "worlds_with_error_flags": float((env.state()["err"] != 0).float().mean())})
        del env, obs, vec, ring, dsc
        torch.cuda.empty_cache()
    return {"workload": "80x80 worlds, 128 agents, FOV sweep (BASELINE.json configs[4])", "n_gpus": world_size, "rows": rows}


def bench_ppo(dev, rank, world_size, worlds=1024, T=256, rows=256, minibatches=8):
    """BASELINE configs[3]: full PPO rollout + update with the restated net.py policy, the GPU vector env (goals sampled on
    device), the GAE kernel and ONE NCCL all-reduce of the flat gradient per minibatch (reference: driver.py:76-134,
    model.py:177-185).  Also checks, over NCCL, that the N-rank gradient of a fixed global minibatch equals the 1-rank
    gradient of the same minibatch (fp32, TF32 off, dropout off): max |g_N - g_1| / max |g_1|."""
    import torch
    import torch.distributed as dist
    from primal_ppo_b200 import BatchedMapfGym, generate_scenario_device
    from primal_ppo_b200.ppo import PPOConfig, ScrimpPolicy, VecPPOTrainer
    group = dist.group.WORLD if world_size > 1 else None
    N = N_AGENTS
    dsc = generate_scenario_device(worlds, H, WD, N, kind="density", density=(0.0, 0.3), queue_len=1, seed=4242,
                                   world_offset=rank * worlds, device=dev)
    env = BatchedMapfGym(dsc, device=dev, seed=1234, use_tape=False, world_offset=rank * worlds, goal_sampling=True)
    torch.manual_seed(0)                                   # identical initial weights on every rank
    pol = ScrimpPolicy().to(dev).use_channels_last()
    cfg = PPOConfig(n_steps=T, n_epochs=1)
    tr = VecPPOTrainer(env, pol, cfg, group=group, amp_dtype=torch.bfloat16, rows_per_minibatch=rows, seed=1234 + rank)

    def sync():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
    # warm-up: a few policy forwards + env steps (cuDNN autotune, allocator), then one timed full rollout
    b = tr.buf
    for t in range(3):
        tr._forward(b.obs[0], b.vec[0], b.ps[0], b.values[0], b.cost_values[0])
    sync()
    t0 = time.perf_counter(); perf = tr.collect(); sync()
    t_roll = _max_over_ranks(time.perf_counter() - t0, dev, world_size)
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for t in range(T):
        env.step_observe(b.actions[t], obs_out=(b.obs[t + 1], b.vec[t + 1]))
    e.record(); torch.cuda.synchronize(dev)
    env_ms = a.elapsed_time(e) / T
    tr.update(perf, max_minibatches=2)                     # warm-up
    sync()
    t0 = time.perf_counter(); stats = tr.update(perf, max_minibatches=minibatches); sync()
    t_upd = _max_over_ranks(time.perf_counter() - t0, dev, world_size)
    out = {"workload": f"PPO rollout+update (BASELINE.json configs[3]): {worlds} worlds/GPU 40x40, {N} agents, T={T}, goals sampled on "
                       f"device, ScrimpPolicy {tr.learner.flat_grad.numel()} params bf16 autocast, minibatch {rows} rows x {N} agents per GPU",
           "n_gpus": world_size, "rollout_agent_steps_per_s": worlds * N * T * world_size / t_roll,
           "rollout_ms_per_step": 1e3 * t_roll / T, "env_ms_per_step": env_ms,
           "update_agent_rows_per_s": rows * N * len(stats) * world_size / t_upd, "update_ms_per_minibatch": 1e3 * t_upd / len(stats),
           "rollout_plus_update_agent_steps_per_s": worlds * N * T * world_size / (t_roll + t_upd * (T * worlds // rows) / len(stats)),
           "note_rollout_plus_update": "one rollout + ONE epoch over all its rows, the update time extrapolated from the timed minibatches",
           "grad_bytes": tr.learner.flat_grad.numel() * 4, "episode_perf": perf, "last_stats": stats[-1]}
    if world_size > 1:
        a.record()
        for _ in range(10):
            dist.all_reduce(tr.learner.flat_grad)
        e.record(); torch.cuda.synchronize(dev)
        out["grad_allreduce_ms"] = _max_over_ranks(a.elapsed_time(e) / 10, dev, world_size)
        out["grad_allreduce_gbs"] = out["grad_bytes"] / (out["grad_allreduce_ms"] * 1e-3) / 1e9
        # ---- N-rank gradient vs 1-rank gradient on the same global minibatch, over NCCL --------------------------------
        tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
        torch.backends.cudnn.allow_tf32 = False; torch.backends.cuda.matmul.allow_tf32 = False
        lr_, amp = tr.learner, tr.learner.amp_dtype
        pol.eval(); lr_.amp_dtype = None
        try:
            per = max(1, 256 // world_size)                # reference MINIBATCH_SIZE rows in total
            g = torch.Generator(device=dev); g.manual_seed(5 + rank)
            mine = b.minibatch(torch.randperm(T * worlds, generator=g, device=dev)[:per])
            full = {}
            for k, v in mine.items():
                parts = [torch.empty_like(v) for _ in range(world_size)]
                dist.all_gather(parts, v.contiguous())
                full[k] = torch.cat(parts)
            lr_.compute_gradients(mine)                    # shard gradient + NCCL all-reduce
            g_n = lr_.flat_grad.clone()
            lr_.group = None
            lr_.compute_gradients(full)                    # the same global minibatch on one rank
            g_1 = lr_.flat_grad.clone()
            lr_.group = group
            d = torch.stack([(g_n - g_1).abs().max(), g_1.abs().max()])
            dist.all_reduce(d, op=dist.ReduceOp.MAX)
            tol = 2e-4
            out["grad_check"] = {"global_minibatch_rows": per * world_size, "max_abs_diff": float(d[0]), "max_abs_grad": float(d[1]),
                                 "rel": float(d[0] / d[1]), "tolerance_rel": tol, "ok": bool(float(d[0]) <= tol * float(d[1])),
                                 "how": "fp32, TF32 off, dropout off; N-rank = shard losses as shares of the global mean + one NCCL "
                                        "all-reduce of the flat gradient; 1-rank = the all-gathered minibatch on one GPU"}
        finally:
            pol.train(); lr_.amp_dtype = amp; lr_.group = group
            torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32
    del tr, env, pol, dsc
    torch.cuda.empty_cache()
    return out


def cpu_port_throughput(budget_s, worlds, threads, seed=7):
    """agent-steps/s of the oracle (C port of the reference's algorithm) on the host cores: the reference's 5-call step
    + getAllObservations on the same kind of worlds and actions, for ~budget_s seconds."""
    from oracle import OracleMapfGym, build_oracle
    from primal_ppo_b200 import random_actions
    build_oracle()
    sc = build_scenario(worlds, seed)
    env = OracleMapfGym(sc, seed=1234, threads=threads, use_tape=False)
    acts = random_actions(16, worlds, N_AGENTS, seed=seed)
    bufs = env.step_observe(acts[0])                            # warm-up
    t0 = time.perf_counter()
    steps = 0
    while True:
        env.step_observe(acts[steps % 16], bufs)
        steps += 1
        if time.perf_counter() - t0 >= budget_s:
            break
    dt = time.perf_counter() - t0
    return worlds * N_AGENTS * steps / dt, steps, dt


def python_reference(budget_s):
    """The UNMODIFIED Python reference env (baseline/_ref, installed by baseline/install_ref.py where /root/reference exists)
    timed on this box's host cores, one process per core: BASELINE configs[2]'s shape and configs[0]."""
    if budget_s <= 0:
        return {"skipped": "--python-ref-budget 0"}
    try:
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        import cpu_baseline
        if not cpu_baseline.available():
            return {"unavailable": "baseline/_ref not shipped (install: python baseline/install_ref.py in the authoring container)"}
        return {"40x40x32": cpu_baseline.run(40, 32, (0.0, 0.3), budget_s), "10x10x8": cpu_baseline.run(10, 8, (0.2, 0.2), budget_s)}
    except Exception as ex:
        return {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}


def run_reference(args):
    """--impl reference: the CPU implementation of the path alone (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # all host threads this process may use (torchrun exports OMP_NUM_THREADS=1; the oracle takes the count explicitly)
    threads = len(os.sched_getaffinity(0))
    worlds = 32 * threads
    from oracle import OracleMapfGym, build_oracle
    from primal_ppo_b200 import random_actions
    build_oracle()
    sc = build_scenario(worlds, 7)
    env = OracleMapfGym(sc, seed=1234, threads=threads, use_tape=False)
    acts = random_actions(16, worlds, N_AGENTS, seed=7)
    bufs = env.step_observe(acts[0])
    # each bench "step" is a bounded sample: `inner` env steps over `worlds` worlds
    inner = 64
    for w in range(args.warmup):
        for k in range(inner):
            env.step_observe(acts[k % 16], bufs)
    t0 = time.perf_counter()
    for s in range(args.steps):
        for k in range(inner):
            env.step_observe(acts[k % 16], bufs)
    dt = time.perf_counter() - t0
    value = worlds * N_AGENTS * inner * args.steps / dt
    sample = f"{worlds} worlds 40x40x32 agents x {inner} env steps per bench step, {threads} OpenMP threads"
    line = {"impl": "reference", "metric": "agent-steps/sec step+observe (40x40, 32 agents)", "value": value,
            "unit": "agent-steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/i16 state, f32 obs", "data": "synthetic",
            "config": bench_config(args.worlds),
            "notes": {"sample": "the CPU path is timed on a bounded sample of the workload: " + sample},
            "cpu_baseline": {"value": value, "unit": "agent-steps/s", "cores": threads, "kind": "port", "sample": sample,
                             "note": "C/OpenMP restatement of mapf_gym.py (oracle/mapf_oracle.c), pinned bit-exact to the "
                                     "reference; the unmodified Python reference on the same cores is under python_reference"},
            "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    # the Python reference itself on the same cores (its own implementation of the same path, ~1e3 agent-steps/s per core):
    # reported beside the port, which is the arm the driver's ratio is computed against
    line["python_reference"] = python_reference(args.python_ref_budget)
    pr = line["python_reference"].get("40x40x32", {}) if isinstance(line["python_reference"], dict) else {}
    if pr.get("agent_steps_per_s"):
        line["cpu_baseline"]["port_vs_python_reference"] = value / pr["agent_steps_per_s"]
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--worlds", type=int, default=65536, help="worlds per GPU")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU-baseline sampling (rank 0, N=1)")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--no-ppo", action="store_true", help="skip the configs[3] PPO rollout+update extra")
    ap.add_argument("--ppo-worlds", type=int, default=1024, help="worlds per GPU of the PPO extra")
    ap.add_argument("--ppo-steps", type=int, default=256, help="rollout length T of the PPO extra")
    ap.add_argument("--sustained-seconds", type=float, default=2.0)
    ap.add_argument("--python-ref-budget", type=float, default=8.0, help="seconds per config of Python-reference timing")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference has none")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from primal_ppo_b200 import BatchedMapfGym, gae
    from primal_ppo_b200.build import build
    build()

    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=dev)
    Wn, N = args.worlds, N_AGENTS
    K, Wu = args.steps, max(args.warmup, 3)

    sc, ring = bench_inputs(Wn, dev, rank)
    env = BatchedMapfGym(sc, device=dev, seed=1234 + rank, use_tape=False)
    obs = torch.empty((Wn, N, CH, FOV, FOV), dtype=torch.float32, device=dev)     # the policy's input tensors
    vec = torch.empty((Wn, N, 4), dtype=torch.float32, device=dev)
    env.getAllObservations(out=(obs, vec))

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ONE pinned slab: 2 result slots + the runner's action ring.  Compact wire format: all per-agent results of a step in
    # 2 bytes per agent (lossless; mapf_decode_results_host expands them) — 4.5 MB instead of 25 MB per step and GPU, which
    # is what keeps eight GPUs of one box below the host's PCIe / memory ceiling (the full f32 slab is timed as an extra)
    ring_h = env.make_host_ring(slots=2, action_slots=8, compact=True)
    for k, r in enumerate(ring):
        ring_h["action_ring"][k].copy_(r)
    host_ring = [ring_h["action_ring"][k] for k in range(8)]

    def run_e2e(n_calls, ring_h=ring_h, sync_ranks=True):
        """n_calls env steps through the split-phase host call, wall clock, after 3 untimed calls.  Every step: the joint
        action is read from pinned host memory (H2D inside the call), ONE fused launch, the step's per-agent results come
        back with one D2H copy and are READ ON THE HOST — one step behind the launch, which is how a rollout loop consumes
        them (runner.py:84-99 only appends them).  Returns (seconds, h2d bytes, d2h bytes per step)."""
        acts_h = ring_h["action_ring"]
        for i in range(3):
            env.step_observe_host_begin(acts_h[i % 8], ring_h["slots"][i & 1], obs, vec)
        env.host_wait(0)
        if sync_ranks:
            barrier()
        else:
            torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        stamps = []
        sink = 0.0
        for i in range(n_calls):
            h2d_, d2h_ = env.step_observe_host_begin(acts_h[i % 8], ring_h["slots"][(i + 3) & 1], obs, vec)
            if i > 0:
                env.host_wait(1)                                         # step i-1 has landed while step i runs
                sink += read_reward(ring_h["slots"][(i + 2) & 1])
            stamps.append(time.perf_counter())
        env.host_wait(0)
        sink += read_reward(ring_h["slots"][(n_calls + 2) & 1])
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        if os.environ.get("BENCH_E2E_DEBUG"):
            d = [round((b - a) * 1e3, 3) for a, b in zip([t0] + stamps[:-1], stamps)]
            print("e2e per-call ms:", d, "mean", round(dt / n_calls * 1e3, 3), file=sys.stderr)
        return dt, h2d_, d2h_

    def read_reward(slot):
        """The host reads a result of the step: agent (0, 0)'s reward, decoded from the packed record in compact mode."""
        if "packed" in slot:
            p = int(slot["packed"][0, 0]) & 0xffff
            return (-2.0, -2.0, -2.0, -0.35, -0.3)[min(p & 7, 4)] + (1.5 if p & 8 else 0.0)
        return float(slot["reward"][0, 0])

    def run_e2e_sync(n_calls):
        """The synchronous form (mapf_step_observe_host: results on the host before the call returns)."""
        hb = env.make_host_buffers(with_obs=False)
        for i in range(3):
            env.step_observe_host(hb, obs, vec, actions=host_ring[i % 8])
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for i in range(n_calls):
            env.step_observe_host(hb, obs, vec, actions=host_ring[i % 8])
            _ = float(hb["reward"][0, 0])
        return time.perf_counter() - t0

    # ---------------- device-resident throughput (value): one fused step+observe launch per step ------------------
    clk = ClockSampler(local_rank).start()          # running before the warm-up so that it has samples in the timed region
    for i in range(Wu):
        env.step_observe(ring[i % 8], obs_out=(obs, vec))
    barrier()
    with clk:
        t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
        t_start.record()
        for i in range(K):
            last = env.step_observe(ring[i % 8], obs_out=(obs, vec))
        t_end.record()
        barrier()
    if args.dump_outputs and rank == 0:           # before the sections below step the env again
        dump_outputs(args.dump_outputs, last)
    total_ms = t_start.elapsed_time(t_end)
    # the dominant kernel's average launch duration over the timed region: K back-to-back launches between two CUDA events
    # on the launching stream (one launch per step and nothing else in between)
    fused_ms = total_ms / K
    tmax = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world_size > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    total_ms_max = float(tmax.item())
    value = Wn * N * K * world_size / (total_ms_max * 1e-3)
    err_frac = float((env.state()["err"] != 0).float().mean())

    # ---------------- the same work as two launches (mapf_step, mapf_observe): per-kernel CUDA-event timings ------
    Kk = max(3, min(K, 20))
    evk = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(Kk)]
    for i in range(3):
        env.step(ring[i % 8]); env.getAllObservations(out=(obs, vec))
    torch.cuda.synchronize(dev)
    for i in range(Kk):
        evk[i][0].record()
        env.step(ring[i % 8])
        evk[i][1].record()
        env.getAllObservations(out=(obs, vec))
        evk[i][2].record()
    torch.cuda.synchronize(dev)
    step_ms = float(np.mean([e[0].elapsed_time(e[1]) for e in evk]))
    obs_ms = float(np.mean([e[1].elapsed_time(e[2]) for e in evk]))

    # ---------------- end to end through the host-buffer C-ABI call ---------------------------------------------
    Ke = max(3, min(K, 50))
    e2e_s, h2d, d2h = run_e2e(Ke)
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world_size > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = Wn * N * Ke * world_size / float(te.item())

    # ---------------- the same device-resident loop held for >= 2 s (does the 20-step number survive?) -------------
    sustained = None
    if not args.no_extras:
        n_sus = int(max(200, args.sustained_seconds * 1e3 / max(fused_ms, 1e-3)))
        clk2 = ClockSampler(local_rank).start()
        barrier()
        with clk2:
            sa, sb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            sa.record()
            for i in range(n_sus):
                env.step_observe(ring[i % 8], obs_out=(obs, vec))
            sb.record()
            barrier()
        sus_ms = _max_over_ranks(sa.elapsed_time(sb), dev, world_size)
        sustained = {"steps": n_sus, "seconds": sus_ms * 1e-3, "ms_per_step": sus_ms / n_sus,
                     "value": Wn * N * n_sus * world_size / (sus_ms * 1e-3), "unit": "agent-steps/s", "clocks": clk2.summary()}

    # ---------------- extras every rank takes part in: strong scaling, configs[4], configs[3] ------------------------
    multi = {}
    if not args.no_extras:
        for name, fn in (("strong", lambda: bench_strong(sc, dev, rank, world_size, max(K, 50))),
                         ("fov_sweep", lambda: bench_fov_sweep(dev, rank, world_size)),
                         ("ppo", lambda: bench_ppo(dev, rank, world_size, worlds=args.ppo_worlds, T=args.ppo_steps))):
            if name == "ppo" and args.no_ppo:
                continue
            try:
                multi[name] = fn()
            except Exception as ex:                      # an extra must never take the headline line down with it
                import traceback
                traceback.print_exc()
                multi[name] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
                torch.cuda.empty_cache()

    line_extra = {}
    if rank == 0 and not args.no_extras:
        try:
            full = env.make_host_ring(slots=2, action_slots=8, compact=False)
            for k, r in enumerate(ring):
                full["action_ring"][k].copy_(r)
            fs, fh, fd = run_e2e(min(Ke, 20), full, sync_ranks=False)
            line_extra["e2e_full_f32_slab"] = {"value": Wn * N * min(Ke, 20) / fs, "unit": "agent-steps/s (this rank)",
                                               "d2h_bytes_per_step": fd,
                                               "note": "the same split-phase call with the 12-byte-per-agent result slab"}
            del full
        except Exception as ex:
            line_extra["e2e_full_f32_slab"] = {"error": str(ex)[:200]}
        try:
            line_extra["e2e_synchronous_call"] = {"value": Wn * N * 10 / run_e2e_sync(10), "unit": "agent-steps/s (1 GPU)",
                                                  "note": "mapf_step_observe_host: results on the host before the call returns"}
        except Exception as ex:
            line_extra["e2e_synchronous_call"] = {"error": str(ex)[:200]}
        # observations copied to host as well (what the reference's getAllObservations returns): PCIe-bound
        try:
            hbo = env.make_host_buffers(with_obs=True)
            hbo["actions"].copy_(host_ring[0]); env.step_observe_host(hbo, obs, vec)
            t0 = time.perf_counter()
            for i in range(2):
                hbo["actions"].copy_(host_ring[i % 8]); _, d2h_full = env.step_observe_host(hbo, obs, vec)
            dt = time.perf_counter() - t0
            line_extra["e2e_obs_to_host"] = {"value": Wn * N * 2 / dt, "unit": "agent-steps/s (1 GPU)",
                                             "d2h_bytes_per_step": d2h_full, "note": "obs+vec also copied to pinned host memory"}
            del hbo
        except Exception as ex:   # host memory for 4 GB pinned buffers may be unavailable
            line_extra["e2e_obs_to_host"] = {"error": str(ex)[:200]}
        # BFS maps (all W*N maps of a reset) and GAE (T=256) with their own algorithmic-byte rooflines
        peak, _ = measured_peaks()
        # context for a write-only kernel: how fast a plain device fill of 4 GiB runs on this GPU
        buf = torch.empty(1 << 30, dtype=torch.float32, device=dev)
        buf.zero_(); torch.cuda.synchronize(dev)
        fa, fb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fa.record()
        for _ in range(5):
            buf.zero_()
        fb.record(); torch.cuda.synchronize(dev)
        line_extra["write_only_fill_gbs"] = 5 * buf.numel() * 4 / (fa.elapsed_time(fb) * 1e-3) / 1e9
        del buf
        nb = min(Wn, 8192)
        ids = torch.arange(nb * N, device=dev, dtype=torch.int32)
        bfs_out = torch.empty((nb * N, H, WD), dtype=torch.int16, device=dev)
        env.bfs_maps(agent_ids=ids, out=bfs_out); torch.cuda.synchronize(dev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(3):
            env.bfs_maps(agent_ids=ids, out=bfs_out)
        b.record(); torch.cuda.synchronize(dev)
        bfs_ms = a.elapsed_time(b) / 3
        bfs_bytes = nb * N * (2 * H * WD + H * WD / N)
        line_extra["bfs"] = {"maps": nb * N, "ms": bfs_ms, "maps_per_s": nb * N / (bfs_ms * 1e-3),
                             "achieved_gbs": bfs_bytes / (bfs_ms * 1e-3) / 1e9, "frac": bfs_bytes / (bfs_ms * 1e-3) / 1e9 / peak}
        del bfs_out
        # SURVEY 8d: BFS "all W*N maps" (reset-time) and "arrivals only" (in-loop mapf_bfs_refresh after a step)
        try:
            maps = env.bfs_maps()                                   # [W, N, H, Wd] int16
            torch.cuda.synchronize(dev)
            a.record(); env.bfs_maps(out=maps); b.record(); torch.cuda.synchronize(dev)
            all_ms = a.elapsed_time(b)
            evr = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(10)]
            arrived = torch.zeros((), dtype=torch.int64, device=dev)
            for i in range(10):
                so = env.step(ring[i % 8])
                arrived += so.goals_reached.sum()
                evr[i][0].record(); env.refresh_bfs(maps); evr[i][1].record()
            torch.cuda.synchronize(dev)
            line_extra["bfs_all_and_refresh"] = {"all_maps": Wn * N, "all_maps_ms": all_ms,
                                                 "refresh_ms_per_step": float(np.mean([x.elapsed_time(y) for x, y in evr])),
                                                 "arrivals_per_step": float(arrived.item()) / 10}
            del maps
        except Exception as ex:
            line_extra["bfs_all_and_refresh"] = {"error": str(ex)[:200]}
        T, cols = 256, 8192 * N
        r = torch.randn((T, cols), device=dev); v = torch.randn((T, cols), device=dev); lv = torch.randn((cols,), device=dev)
        gae(r, v, lv); torch.cuda.synchronize(dev)
        a.record()
        for _ in range(3):
            gae(r, v, lv)
        b.record(); torch.cuda.synchronize(dev)
        gae_ms = a.elapsed_time(b) / 3
        gae_bytes = 12.0 * T * cols
        line_extra["gae"] = {"T": T, "cols": cols, "ms": gae_ms, "elements_per_s": T * cols / (gae_ms * 1e-3),
                             "achieved_gbs": gae_bytes / (gae_ms * 1e-3) / 1e9, "frac": gae_bytes / (gae_ms * 1e-3) / 1e9 / peak}
        try:                      # both rollout streams (rewards / values, costRewards / costValues) in ONE launch: mapf_gae2
            from primal_ppo_b200 import gae2
            cr = torch.randn((T, cols), device=dev); cv = torch.randn((T, cols), device=dev)
            gae2(r, v, lv, cr, cv, lv); torch.cuda.synchronize(dev)
            a.record()
            for _ in range(3):
                gae2(r, v, lv, cr, cv, lv)
            b.record(); torch.cuda.synchronize(dev)
            g2 = a.elapsed_time(b) / 3
            line_extra["gae"].update(two_streams_ms=g2, two_streams_gbs=2 * gae_bytes / (g2 * 1e-3) / 1e9,
                                     two_streams_frac=2 * gae_bytes / (g2 * 1e-3) / 1e9 / peak)
            del cr, cv
        except Exception as ex:
            line_extra["gae"]["two_streams_error"] = str(ex)[:200]
        del r, v, lv
        # optional bf16 observation format (same values, half the bytes; not the reference layout, not the headline)
        try:
            ob16 = torch.empty((Wn, N, CH, FOV, FOV), dtype=torch.bfloat16, device=dev)
            for i in range(3):
                env.step_observe(ring[i % 8], obs_out=(ob16, vec))
            torch.cuda.synchronize(dev)
            a.record()
            for i in range(10):
                env.step_observe(ring[i % 8], obs_out=(ob16, vec))
            b.record(); torch.cuda.synchronize(dev)
            ms16 = a.elapsed_time(b) / 10
            line_extra["bf16_observations"] = {"ms_per_step": ms16, "agent_steps_per_s": Wn * N / (ms16 * 1e-3),
                                               "note": "mapf_step_observe_bf16: optional output format, outside the reference layout"}
            del ob16
        except Exception as ex:
            line_extra["bf16_observations"] = {"error": str(ex)[:200]}
        # reset-time work (not on the step path): on-device generation of 65 536 worlds, mapf_reset
        try:
            from primal_ppo_b200 import generate_scenario_device
            nw = min(Wn, 65536)
            generate_scenario_device(256, H, WD, N, kind="density", density=(0.0, 0.3), queue_len=16, seed=1, device=dev)
            torch.cuda.synchronize(dev)
            a.record()
            dsc = generate_scenario_device(nw, H, WD, N, kind="density", density=(0.0, 0.3), queue_len=16, seed=2, device=dev)
            b.record(); torch.cuda.synchronize(dev)
            gen_ms = a.elapsed_time(b)
            a.record(); env.reset(); b.record(); torch.cuda.synchronize(dev)
            line_extra["reset"] = {"worlds": nw, "generate_scenario_ms": gen_ms, "mapf_reset_ms": a.elapsed_time(b),
                                   "generator_flagged_worlds": float(((dsc.gen_err & ~4) != 0).float().mean())}
            del dsc
        except Exception as ex:
            line_extra["reset"] = {"error": str(ex)[:200]}

    if rank == 0:
        peak, peak_src = measured_peaks()
        b_step, b_obs, b_fused = algorithmic_bytes()
        obs_bytes = b_obs * Wn * N
        step_bytes = b_step * Wn * N
        fused_bytes = b_fused * Wn * N
        achieved = fused_bytes / (fused_ms * 1e-3) / 1e9
        cpu = None
        if world_size == 1 and args.cpu_budget > 0:
            threads = len(os.sched_getaffinity(0))
            cw = 32 * threads
            cv, csteps, cdt = cpu_port_throughput(args.cpu_budget, cw, threads)
            cpu = {"value": cv, "unit": "agent-steps/s", "cores": threads, "kind": "port",
                   "sample": f"{cw} worlds 40x40x32 agents, {csteps} steps in {cdt:.1f} s, {threads} OpenMP threads (oracle/mapf_oracle.c)"}
            if not args.no_extras and args.python_ref_budget > 0:
                cpu["python_reference"] = python_reference(args.python_ref_budget)
        line = {"metric": "agent-steps/sec step+observe (40x40, 32 agents)", "value": value, "unit": "agent-steps/s",
                "n_gpus": world_size, "steps": K, "warmup": Wu, "ms_per_step": total_ms_max / K, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8/i16 state, f32 obs", "data": "synthetic",
                "config": bench_config(Wn),
                "notes": {"actions": "uniform random, device-resident ring of 8",
                          "call": "mapf_step_observe (one fused launch per step)",
                          "l2": "working set per step (obs 4.08 GB/GPU written) far exceeds the 126 MB L2; no flush needed",
                          "worlds_with_error_flags": err_frac},
                "clocks": clk.summary(),
                "e2e": {"value": e2e_value, "unit": "agent-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "steps": Ke, "note": "mapf_step_observe_host_begin/_wait (split-phase, compact wire format): every step the joint "
                                             "action comes from pinned host memory (H2D), ONE fused launch, and ALL per-agent results "
                                             "(status, reward, cost, goals reached, violations, executed actions: 16 bits per agent, "
                                             "lossless, + shadow goals) return in one D2H copy and are read on the host one step behind "
                                             "the launch; "
                                             "observations and trainValid stay in HBM as the policy's / learner's input tensors"},
                "gpu_launches": K,
                "roofline": {"bound": "hbm", "kernel": "step_observe_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                             "frac": achieved / peak, "traffic": ncu_traffic("step_observe_kernel"), "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": fused_bytes, "ms_per_launch": fused_ms,
                             "algorithmic_bytes_per_agent_step": b_fused},
                "kernels": {"step_observe_kernel": {"ms": fused_ms, "algorithmic_bytes": fused_bytes, "achieved_gbs": achieved,
                                                    "frac": achieved / peak, "traffic": ncu_traffic("step_observe_kernel")},
                            "step_kernel": {"ms": step_ms, "algorithmic_bytes": step_bytes,
                                            "achieved_gbs": step_bytes / (step_ms * 1e-3) / 1e9,
                                            "frac": step_bytes / (step_ms * 1e-3) / 1e9 / peak,
                                            "traffic": ncu_traffic("step_kernel")},
                            "observe_kernel": {"ms": obs_ms, "algorithmic_bytes": obs_bytes,
                                               "achieved_gbs": obs_bytes / (obs_ms * 1e-3) / 1e9,
                                               "frac": obs_bytes / (obs_ms * 1e-3) / 1e9 / peak,
                                               "traffic": ncu_traffic("observe_kernel")},
                            "note": "step_kernel / observe_kernel: the same work as two launches (mapf_step, mapf_observe), "
                                    "timed in a separate loop of %d steps" % Kk},
                "cpu_baseline": cpu}
        if sustained is not None:
            line["sustained"] = sustained
        line.update(multi)
        line.update(line_extra)
        print(json.dumps(line), flush=True)
    if world_size > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
