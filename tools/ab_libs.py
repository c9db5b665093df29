#!/usr/bin/env python
"""In-process A/B of two BUILDS of the library (e.g. before / after a state-layout change): both .so files are loaded,
one env per build on the same tensors, interleaved rounds.   python tools/ab_libs.py tools/_base_libmapf.so"""
import os, sys
import numpy as np
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import primal_ppo_b200._cabi as cabi
from primal_ppo_b200 import BatchedMapfGym, random_scenario
other = os.path.abspath(sys.argv[1])
W, N = 65536, 32
sc = random_scenario(W, 40, 40, N, density=(0.0, 0.3), queue_len=16, seed=100, unique_maps=256)
envs = {"new": BatchedMapfGym(sc, use_tape=False)}
import ctypes


class _OlderBuild(ctypes.CDLL):
    """A build from before some entry points existed: the binding's missing names become inert stubs (never called here)."""
    def __getattr__(self, name):
        try:
            return super().__getattr__(name)
        except AttributeError:
            if name.startswith("__"):
                raise
            stub = type("MissingEntryPoint", (), {})()
            setattr(self, name, stub)
            return stub


cabi._lib = None; cabi.LIB_PATH = other
_cdll, ctypes.CDLL = ctypes.CDLL, _OlderBuild
envs["base"] = BatchedMapfGym(sc, use_tape=False)
ctypes.CDLL = _cdll
dev = envs["new"].device
obs = torch.empty((W, N, 6, 9, 9), device=dev); vec = torch.empty((W, N, 4), device=dev)
gen = torch.Generator(device=dev); gen.manual_seed(1)
ring = [torch.randint(0, 5, (W, N), generator=gen, device=dev, dtype=torch.int8) for _ in range(8)]
res = {k: {"fused": [], "observe": [], "step": [], "two": []} for k in envs}
for rnd in range(7):
    for name, e in envs.items():
        for key, fn in (("fused", lambda i: e.step_observe(ring[i % 8], obs_out=(obs, vec))),
                        ("observe", lambda i: e.getAllObservations(out=(obs, vec))), ("step", lambda i: e.step(ring[i % 8])),
                        ("two", lambda i: (e.step(ring[i % 8]), e.getAllObservations(out=(obs, vec))))):
            for i in range(3):
                fn(i)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for i in range(20):
                fn(i)
            b.record(); torch.cuda.synchronize()
            if rnd:
                res[name][key].append(a.elapsed_time(b) / 20)
for name in envs:
    print(f"{name:5s} " + " ".join(f"{k}={np.median(v):.4f}" for k, v in res[name].items()), flush=True)
# both builds must agree on the state they reached (same scenario, same actions)
s1, s2 = envs["new"].state(), envs["base"].state()
print("states equal:", all(torch.equal(s1[k], s2[k]) for k in s1), "counters equal:", torch.equal(envs["new"].counters(), envs["base"].counters()))
