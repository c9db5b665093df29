"""Scenarios generated ON the GPU (`mapf_generate_scenario`, csrc/scenario_gen.cu): the throughput-mode replacement of
what `MapfGym.__init__` draws on the host (map, human walk, starts, goals; mapf_gym.py:164-190, map_generator.py).

`DeviceScenario` holds the same arrays as `Scenario` as CUDA tensors; `BatchedMapfGym` accepts either.  `to_host()`
gives the numpy `Scenario` (e.g. to replay the same worlds through the oracle)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Optional

import numpy as np
import torch

from . import _cabi
from .scenario import Scenario


@dataclass
class DeviceScenario:
    obst: torch.Tensor          # u8  [W,H,Wd]
    starts: torch.Tensor        # i16 [W,N,2]
    goal_queue: torch.Tensor    # i16 [W,N,Q,2]
    htrace: torch.Tensor        # i16 [W,L,4]
    hlen: torch.Tensor          # i32 [W]
    dims: Optional[torch.Tensor] = None     # i16 [W,2]
    hp5: Optional[torch.Tensor] = None      # i16 [W,5,2]
    gen_err: Optional[torch.Tensor] = None  # i32 [W] generator flags (see include/mapf_b200.h)
    tape: None = None
    tape_len: None = None
    fov: int = 9
    num_channel: int = 6
    use_da: bool = False
    use_hp: bool = False
    meta: dict = field(default_factory=dict)

    num_worlds = property(lambda s: int(s.obst.shape[0]))
    height = property(lambda s: int(s.obst.shape[1]))
    width = property(lambda s: int(s.obst.shape[2]))
    num_agents = property(lambda s: int(s.starts.shape[1]))

    def validate(self) -> None:
        """Shape / dtype checks (ValueError).  The arrays come from `mapf_generate_scenario`, which only ever emits cells
        inside the world and on free cells; their values are therefore not re-checked here (that would be a host sync)."""
        def need(cond, msg):
            if not cond:
                raise ValueError("DeviceScenario: " + msg)
        W, N = self.num_worlds, self.num_agents
        need(self.obst.dtype == torch.uint8 and self.obst.is_cuda and self.obst.is_contiguous(), "obst must be a contiguous CUDA uint8 tensor")
        need(self.starts.shape == (W, N, 2) and self.starts.dtype == torch.int16, "starts must be int16 [W,N,2]")
        need(self.goal_queue.shape[:2] == (W, N) and self.goal_queue.shape[3] == 2 and self.goal_queue.dtype == torch.int16,
             "goal_queue must be int16 [W,N,Q,2]")
        need(self.htrace.shape[0] == W and self.htrace.shape[2] == 4 and self.htrace.dtype == torch.int16, "htrace must be int16 [W,L,4]")
        need(self.hlen.shape == (W,) and self.hlen.dtype == torch.int32, "hlen must be int32 [W]")
        need(self.fov % 2 == 1 and self.fov >= 3 and self.num_channel in (5, 6), "fov odd >= 3, num_channel 5 or 6")

    def to_host(self) -> Scenario:
        n = lambda t: None if t is None else t.cpu().numpy()
        return Scenario(obst=n(self.obst), starts=n(self.starts), goal_queue=n(self.goal_queue), htrace=n(self.htrace),
                        hlen=n(self.hlen), hp5=n(self.hp5), dims=n(self.dims), fov=self.fov, num_channel=self.num_channel,
                        use_da=self.use_da, use_hp=self.use_hp, meta=dict(self.meta))


def generate_scenario_device(num_worlds: int, height: int, width: int, num_agents: int, *, kind: str = "density",
                             density=(0.0, 0.3), triangular: bool = False, size_range=None, queue_len: int = 16,
                             trace_len: Optional[int] = None, human_loops: int = 1, seed: int = 0, world_offset: int = 0,
                             device=None, fov: int = 9, num_channel: int = 6, use_da: bool = False,
                             use_hp: bool = False, human_path: str = "bfs") -> DeviceScenario:
    """kind="warehouse": `generateWarehouse(num_block=size_range)` worlds (training env; default size_range (10, 40)
    needs height >= 40, width >= 60).  kind="density": `rand < p` maps, p per world from `density`; `size_range` =
    (lo, hi) draws the side like `random_generator`, None keeps height x width.
    human_path="astar4" walks the human along astar_4's path to each goal, bit-exact with the reference's `MapfGym()`;
    "bfs" (the default) along another shortest path (a BFS descent).  Everything else is the same for both."""
    if not torch.cuda.is_available():
        raise _cabi.MapfError("generate_scenario_device needs a CUDA device; there is no CPU fallback")
    lib = _cabi.load_library()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    W, H, Wd, N, Q = num_worlds, height, width, num_agents, queue_len
    k = {"density": 0, "warehouse": 1}[kind]
    hp = {"bfs": 0, "astar4": 1}[human_path]
    if k == 1 and size_range is None:
        size_range = (10, 40)
    lo, hi = (0, 0) if size_range is None else (int(size_range[0]), int(size_range[1]))
    L = int(trace_len) if trace_len else 2 * (H + Wd) * max(1, human_loops) + 2
    z = lambda *s, dt: torch.empty(s, dtype=dt, device=dev)
    sc = DeviceScenario(obst=z(W, H, Wd, dt=torch.uint8), starts=z(W, N, 2, dt=torch.int16),
                        goal_queue=z(W, N, Q, 2, dt=torch.int16), htrace=z(W, L, 4, dt=torch.int16),
                        hlen=z(W, dt=torch.int32), dims=z(W, 2, dt=torch.int16), hp5=z(W, 5, 2, dt=torch.int16),
                        gen_err=z(W, dt=torch.int32), fov=fov, num_channel=num_channel, use_da=use_da, use_hp=use_hp,
                        meta=dict(kind=kind, density=list(density), size_range=[lo, hi], seed=seed, generator="device",
                                  human_path=human_path))
    cfg = _cabi.MapfGenConfig(num_worlds=W, height=H, width=Wd, num_agents=N, kind=k, density_mode=int(triangular),
                              density_lo=float(density[0]), density_hi=float(density[1]), size_lo=lo, size_hi=hi,
                              queue_len=Q, trace_len=L, human_loops=int(human_loops), human_path=hp,
                              seed=int(seed) & (2 ** 64 - 1),
                              world_offset=int(world_offset), device=dev.index or 0)
    p = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    with torch.cuda.device(dev):
        _cabi.check(lib.mapf_generate_scenario(C.byref(cfg), p(sc.obst), p(sc.dims), p(sc.starts), p(sc.goal_queue),
                                               p(sc.htrace), p(sc.hlen), p(sc.hp5), p(sc.gen_err), stream),
                    "mapf_generate_scenario")
    return sc


def astar_paths_device(obst: torch.Tensor, start_goal: torch.Tensor, max_len: Optional[int] = None):
    """astar_4 paths for n (map, start, goal) triples in one `mapf_astar4_paths` call, bit-exact with
    `episode_io.astar_path`.  obst: CUDA uint8 [n,H,Wd] (nonzero = wall), start_goal: int16 [n,2,2] (row, col) pairs on
    the same device.  Returns (paths i16 [n,max_len,2], lens i32 [n]) on that device: lens k >= 1 is a path of k cells,
    0 start == goal, -1 no path, -2 longer than max_len (default H * Wd, every path fits), -3 a cell outside the map;
    unused path cells are -1.  Asynchronous on the current stream."""
    lib = _cabi.load_library()
    if not (obst.is_cuda and obst.dtype == torch.uint8 and obst.dim() == 3):
        raise ValueError("astar_paths_device: obst must be a CUDA uint8 tensor [n,H,Wd]")
    n, H, Wd = obst.shape
    if start_goal.shape != (n, 2, 2) or start_goal.dtype != torch.int16 or start_goal.device != obst.device:
        raise ValueError("astar_paths_device: start_goal must be int16 [n,2,2] on the device of obst")
    L = H * Wd if max_len is None else int(max_len)
    obst, start_goal = obst.contiguous(), start_goal.contiguous()
    paths = torch.empty((n, max(L, 0), 2), dtype=torch.int16, device=obst.device)
    lens = torch.empty((n,), dtype=torch.int32, device=obst.device)
    if n == 0:
        return paths, lens
    p = lambda t: C.c_void_p(t.data_ptr())
    with torch.cuda.device(obst.device):
        stream = C.c_void_p(torch.cuda.current_stream(obst.device).cuda_stream)
        _cabi.check(lib.mapf_astar4_paths(p(obst), n, H, Wd, p(start_goal), L, p(paths), p(lens), stream), "mapf_astar4_paths")
    return paths, lens
